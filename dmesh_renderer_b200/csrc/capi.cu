// capi.cu -- extern "C" boundary of libdmesh_b200.so (see include/dmesh_b200.h).
// Host-side stage sequencing; replaces CudaRasterizer::Rasterizer::forward /
// backward (cuda_rasterizer/rasterizer_impl.cu:175-383, 387-467) and
// CudaRenderer::Renderer::forward / backward (cuda_renderer/renderer_impl.cu:193-498)
// without their per-stage cudaDeviceSynchronize (auxiliary.h:425-432).
#include "tri.cuh"
#include "tet.cuh"
#include "../../include/dmesh_b200.h"
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <sched.h>

namespace dmr {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
int cuda_fail(cudaError_t e, const char* what)
{
    set_error("CUDA error in %s: %s", what, cudaGetErrorString(e));
    return DMR_ECUDA;
}

// ---- stage timing ------------------------------------------------------------
static const char* const g_stage_names[ST_COUNT] = {
    "preprocess_points", "preprocess_faces", "face_depth_sort", "scan", "duplicate_with_keys", "sort_histogram", "sort_plan",
    "sort_pass0", "sort_pass1", "sort_pass2", "sort_pass3", "sort_pass4", "sort_pass5", "sort_pass6", "sort_pass7",
    "tile_ranges", "tri_render_forward", "tri_render_backward", "tri_grad_finish", "tet_build_records", "tet_jitter",
    "tet_first_intersect", "tet_march_forward", "tet_march_backward", "tet_grad_vertex", "tri_render_backward_camera",
    "tri_camera_finish", "depth_chain_camera", "depth_chain_camera_finish", "tet_march_backward_camera", "tet_camera_finish",
    "tet_march_backward_vertex", "tet_march_backward_camera_vertex", "tet_vertex_finish",
    "tet_march_backward_intensity", "tet_march_backward_camera_intensity", "tet_march_backward_vertex_intensity",
    "tet_march_backward_camera_vertex_intensity", "tet_intensity_finish", "tri_alpha", "tri_render_backward_alpha",
    "tri_background_grad", "tet_alpha", "tet_march_backward_alpha", "tet_background_grad", "tri_face_weights",
    "tet_face_weights" };
struct Prof {
    bool on = false, created = false;
    cudaEvent_t ev[ST_COUNT][2];
    bool used[ST_COUNT];
};
static Prof g_prof;
static unsigned long long g_launches = 0;   // kernels launched by this library (bench.py: gpu_launches)
void count_launch(int n) { g_launches += (unsigned long long)n; }
void prof_begin(int stage, cudaStream_t s, bool count)
{
    if (count) g_launches++;
    if (!g_prof.on) return;
    if (!g_prof.created) {
        for (int i = 0; i < ST_COUNT; i++) { cudaEventCreate(&g_prof.ev[i][0]); cudaEventCreate(&g_prof.ev[i][1]); g_prof.used[i] = false; }
        g_prof.created = true;
    }
    cudaEventRecord(g_prof.ev[stage][0], s);
}
void prof_end(int stage, cudaStream_t s)
{
    if (!g_prof.on) return;
    cudaEventRecord(g_prof.ev[stage][1], s);
    g_prof.used[stage] = true;
}

BinningLayout BinningLayout::make(size_t R)
{
    BinningLayout L;
    size_t o = 0;
    L.keys_unsorted = o; o = align_up(o + 4 * R, 256);
    L.vals_unsorted = o; o = align_up(o + 4 * R, 256);
    L.keys_sorted = o;   o = align_up(o + 4 * R, 256);
    L.vals_sorted = o;   o = align_up(o + 4 * R, 256);
    L.sort_temp = o;     o = align_up(o + sort_temp_bytes_u32(R), 256);
    L.total = o + 256;
    return L;
}

static bool sizes_ok(long long B, long long P, long long F, long long W, long long H)
{
    if (B < 0 || P < 0 || F < 0 || W <= 0 || H <= 0) { set_error("negative or zero size"); return false; }
    if (B * P >= (1LL << 31) || B * F >= (1LL << 31) || B * W * H >= (1LL << 31)) {
        set_error("B*P, B*F and B*W*H must stay below 2^31");
        return false;
    }
    if ((W + DMR_TILE - 1) / DMR_TILE >= 65536 || (H + DMR_TILE - 1) / DMR_TILE >= 65536) {
        set_error("image too large for 16-bit tile coordinates");
        return false;
    }
    return true;
}

// workspace of the camera-gradient backward: the mode's own scratch, then 24 floats per (view, tile)
static size_t tri_cam_bytes(int B, int P, int F, int W, int H, bool deterministic)
{
    const size_t base = deterministic ? TriDetLayout::make((size_t)B, (size_t)P, (size_t)F).total
                                      : TriBwdLayout::make((size_t)B * F, (size_t)P).total;
    const size_t tiles = (size_t)B * ((W + DMR_TILE - 1) / DMR_TILE) * ((H + DMR_TILE - 1) / DMR_TILE);
    return align_up(base, 256) + align_up(96 * tiles, 256) + 256;
}

template <typename T>
static T* at(void* base, size_t off) { return reinterpret_cast<T*>(static_cast<unsigned char*>(base) + off); }
template <typename T>
static const T* at(const void* base, size_t off) { return reinterpret_cast<const T*>(static_cast<const unsigned char*>(base) + off); }

}  // namespace dmr

using namespace dmr;

extern "C" {

int dmr_abi_version(void) { return 2; }
const char* dmr_last_error(void) { return g_err; }

unsigned long long dmr_launch_count(void) { return g_launches; }

int dmr_profile_enable(int on)
{
    g_prof.on = on != 0;
    if (g_prof.created) for (int i = 0; i < ST_COUNT; i++) g_prof.used[i] = false;
    return DMR_OK;
}
int dmr_profile_stage_count(void) { return ST_COUNT; }
const char* dmr_profile_stage_name(int i) { return (i >= 0 && i < ST_COUNT) ? g_stage_names[i] : ""; }
int dmr_profile_read(float* ms_out)
{
    if (!ms_out) { set_error("ms_out is null"); return DMR_EINVAL; }
    for (int i = 0; i < ST_COUNT; i++) {
        ms_out[i] = -1.0f;
        if (!g_prof.created || !g_prof.used[i]) continue;
        cudaError_t e = cudaEventSynchronize(g_prof.ev[i][1]);
        if (e != cudaSuccess) return cuda_fail(e, "cudaEventSynchronize");
        float ms = 0;
        e = cudaEventElapsedTime(&ms, g_prof.ev[i][0], g_prof.ev[i][1]);
        if (e != cudaSuccess) return cuda_fail(e, "cudaEventElapsedTime");
        ms_out[i] = ms;
        g_prof.used[i] = false;
    }
    return DMR_OK;
}

int dmr_wait_i32(volatile int32_t* host_value, int32_t sentinel, dmr_stream_t stream_)
{
    // Poll the pinned word (the D2H copy of num_rendered lands a few microseconds before a
    // cudaStreamSynchronize would return).  The first ~50 us are a tight pause loop (the common case: phase 1 of
    // a small scene is nearly done when the host gets here); after that the thread yields its core between polls,
    // so that several ranks sharing a host do not each burn a core for the whole of a long phase 1.  A finished
    // or faulted stream ends the wait through the stream synchronisation, which also reports the fault.
    if (!host_value) { set_error("host_value is null"); return DMR_EINVAL; }
    for (long long spin = 0; spin < 2000000000LL; spin++) {
        if (*host_value != sentinel) return DMR_OK;
        __builtin_ia32_pause();
        if (spin > 4096) sched_yield();
        if ((spin & 0x3fff) == 0x3fff && cudaStreamQuery((cudaStream_t)stream_) != cudaErrorNotReady) break;
    }
    DMR_CUDA(cudaStreamSynchronize((cudaStream_t)stream_));
    return DMR_OK;
}

int dmr_tri_state_bytes(int B, int P, int F, int W, int H, size_t out[3])
{
    if (!out) { set_error("out is null"); return DMR_EINVAL; }
    if (!sizes_ok(B, P, F, W, H)) return DMR_ETOOLARGE;
    out[0] = align_up(sizeof(float4) * (size_t)B * P, 256) + 256;
    out[1] = TriFaceLayout::make((size_t)B * F).total;
    out[2] = TriImageLayout::make(B, W, H).total;
    return DMR_OK;
}

size_t dmr_binning_bytes(size_t R) { return BinningLayout::make(R).total; }

size_t dmr_sort_temp_bytes(size_t n) { return sort_temp_bytes(n); }

int dmr_sort_pairs(const uint64_t* keys_in, const uint32_t* vals_in, uint64_t* keys_out, uint32_t* vals_out, size_t n,
                   int end_bit, void* temp, dmr_stream_t stream)
{
    if (n && (!keys_in || !vals_in || !keys_out || !vals_out || !temp)) { set_error("null pointer"); return DMR_EINVAL; }
    return sort_pairs(keys_in, vals_in, keys_out, vals_out, n, end_bit, temp, (cudaStream_t)stream);
}

int dmr_sort_pairs_u32(const uint32_t* keys_in, const uint32_t* vals_in, uint32_t* keys_out, uint32_t* vals_out, size_t n,
                       int end_bit, void* temp, dmr_stream_t stream)
{
    if (n && (!keys_in || !keys_out || !vals_out || !temp)) { set_error("null pointer"); return DMR_EINVAL; }
    return sort_pairs_u32(keys_in, vals_in, keys_out, vals_out, n, end_bit, temp, true, (cudaStream_t)stream);
}

int dmr_tri_forward_bin(int B, int P, int F, int W, int H, const float* verts, const int* faces,
                        const float* verts_color, const float* faces_opacity, const float* mv_mats,
                        const float* proj_mats, const float* verts_depth, const float* faces_intense,
                        void* point_buffer, void* face_buffer, int32_t* num_rendered_host, dmr_stream_t stream_)
{
    cudaStream_t stream = (cudaStream_t)stream_;
    if (!sizes_ok(B, P, F, W, H)) return DMR_ETOOLARGE;
    if (!num_rendered_host) { set_error("num_rendered_host is null"); return DMR_EINVAL; }
    if (B == 0 || P == 0 || F == 0) { *num_rendered_host = 0; return DMR_OK; }
    // verts_depth == NULL selects the fused vertex depth (the vertex's own NDC z, dmr_tri_depth_chain in backward)
    if (!verts || !faces || !verts_color || !faces_opacity || !mv_mats || !proj_mats ||
        !faces_intense || !point_buffer || !face_buffer) { set_error("null pointer"); return DMR_EINVAL; }
    const size_t BF = (size_t)B * F;
    TriFaceLayout L = TriFaceLayout::make(BF);
    float4* vimg = static_cast<float4*>(point_buffer);
    int rc;
    SortPre face_sort;
    if ((rc = bin_faces_begin(BF, face_buffer, L.bin, &face_sort, stream))) return rc;
    if ((rc = preprocess_points(B, P, W, H, verts, mv_mats, proj_mats, verts_depth, 1, vimg, stream))) return rc;
    if ((rc = tri_preprocess_faces(B, P, F, W, H, faces, vimg, verts, verts_color, faces_opacity, faces_intense,
                                   at<uint32_t>(face_buffer, L.bin.tiles_touched), at<uint32_t>(face_buffer, L.bin.depth_key),
                                   at<uint2>(face_buffer, L.bin.rect), at<TriRecord>(face_buffer, L.records), face_sort,
                                   stream)))
        return rc;
    return bin_faces(BF, face_buffer, L.bin, num_rendered_host, stream);
}

int dmr_tri_depth_chain(int B, int P, const float* verts, const float* mv_mats, const float* proj_mats,
                        const float* dL_dvdepth, float* dL_dverts, dmr_stream_t stream)
{
    if (B < 0 || P < 0) { set_error("negative size"); return DMR_EINVAL; }
    if (B == 0 || P == 0) return DMR_OK;
    if (!verts || !mv_mats || !proj_mats || !dL_dvdepth || !dL_dverts) { set_error("null pointer"); return DMR_EINVAL; }
    return depth_chain(B, P, verts, mv_mats, proj_mats, dL_dvdepth, dL_dverts, (cudaStream_t)stream);
}

// phase 2; face_weights != nullptr: also the face statistics (face_weights, face_hits, workspace checked by the caller)
static int tri_forward_render_impl(int B, int P, int F, int W, int H, int R, const float* background,
                                   const float* inv_mv_mats, const float* inv_proj_mats, const void* point_buffer,
                                   void* face_buffer, void* binning_buffer, void* image_buffer, float* out_color,
                                   float* out_depth, dmr_stream_t stream_, float* face_weights = nullptr,
                                   int* face_hits = nullptr, void* workspace = nullptr)
{
    cudaStream_t stream = (cudaStream_t)stream_;
    if (!sizes_ok(B, P, F, W, H) || R < 0) return DMR_ETOOLARGE;
    if (B == 0) return DMR_OK;
    if (!background || !inv_mv_mats || !inv_proj_mats || !image_buffer || !out_color || !out_depth ||
        (R > 0 && (!binning_buffer || !face_buffer))) { set_error("null pointer"); return DMR_EINVAL; }
    (void)point_buffer;
    FaceWeightAcc fw{};
    if (face_weights) {
        // zeroed before every phase 2: a call repeated after a too-small speculative binning buffer starts afresh
        fw = face_weights_acc(workspace, B, F);
        DMR_CUDA(cudaMemsetAsync(workspace, 0, face_weights_bytes(B, F), stream));
    }
    TriFaceLayout FL = TriFaceLayout::make((size_t)B * F);
    TriImageLayout IL = TriImageLayout::make(B, W, H);
    uint2* ranges = at<uint2>(image_buffer, IL.ranges);
    int rc = bin_instances(B, F, W, H, (size_t)R, face_buffer, FL.bin, binning_buffer, ranges, stream);
    if (rc) return rc;
    TriRenderParams p = {};
    p.B = B; p.F = F; p.W = W; p.H = H; p.P = P;
    p.ranges = ranges;
    if (R) {
        BinningLayout BL = BinningLayout::make((size_t)R);
        p.face_list = at<uint32_t>(binning_buffer, BL.vals_sorted);
        p.records = at<TriRecord>(face_buffer, FL.records);
    }
    p.bg = background; p.inv_mv = inv_mv_mats; p.inv_proj = inv_proj_mats;
    p.final_T = at<float>(image_buffer, IL.final_T);
    p.prev_T = at<float>(image_buffer, IL.prev_T);
    p.n_contrib = at<uint32_t>(image_buffer, IL.n_contrib);
    p.out_color = out_color; p.out_depth = out_depth;
    if (!face_weights) return tri_render_forward(p, stream);
    if ((rc = tri_render_forward(p, stream, &fw))) return rc;
    ProfScope prof(ST_TRI_FACE_WEIGHTS, stream);
    return face_weights_convert(B, F, fw, face_weights, face_hits, stream);
}

int dmr_tri_forward_render(int B, int P, int F, int W, int H, int R, const float* background,
                           const float* inv_mv_mats, const float* inv_proj_mats, const void* point_buffer,
                           void* face_buffer, void* binning_buffer, void* image_buffer, float* out_color,
                           float* out_depth, dmr_stream_t stream)
{
    return tri_forward_render_impl(B, P, F, W, H, R, background, inv_mv_mats, inv_proj_mats, point_buffer, face_buffer,
                                   binning_buffer, image_buffer, out_color, out_depth, stream);
}

size_t dmr_tri_face_weights_bytes(int B, int F) { return (B < 0 || F < 0) ? 0 : face_weights_bytes(B, F); }

int dmr_tri_forward_render_face_weights(int B, int P, int F, int W, int H, int R, const float* background,
                                        const float* inv_mv_mats, const float* inv_proj_mats, const void* point_buffer,
                                        void* face_buffer, void* binning_buffer, void* image_buffer, float* out_color,
                                        float* out_depth, float* face_weights, int* face_hits, void* workspace,
                                        size_t workspace_bytes, dmr_stream_t stream)
{
    if (!sizes_ok(B, P, F, W, H) || R < 0) return DMR_ETOOLARGE;
    if ((long long)W * H >= (1LL << 31)) { set_error("face statistics need fewer than 2^31 pixels per view"); return DMR_ETOOLARGE; }
    if ((size_t)B * F == 0)   // [B,0] statistics: nothing to count, but the images and the image state as without them
        return tri_forward_render_impl(B, P, F, W, H, R, background, inv_mv_mats, inv_proj_mats, point_buffer, face_buffer,
                                       binning_buffer, image_buffer, out_color, out_depth, stream);
    if (!face_weights || !face_hits) { set_error("null pointer: face_weights / face_hits"); return DMR_EINVAL; }
    const size_t need = face_weights_bytes(B, F);
    if (!workspace || workspace_bytes < need) {
        set_error("face statistics need a workspace of %zu bytes (dmr_tri_face_weights_bytes)", need);
        return DMR_EINVAL;
    }
    return tri_forward_render_impl(B, P, F, W, H, R, background, inv_mv_mats, inv_proj_mats, point_buffer, face_buffer,
                                   binning_buffer, image_buffer, out_color, out_depth, stream, face_weights, face_hits,
                                   workspace);
}

static int tri_backward_impl(int B, int P, int F, int W, int H, int R, const float* background, const float* inv_mv_mats,
                             const float* inv_proj_mats, const void* point_buffer, const void* face_buffer,
                             const void* binning_buffer, const void* image_buffer, const float* dL_dcolor,
                             const float* dL_ddepth, float* dL_dverts, float* dL_dvcolor, float* dL_dfopacity,
                             float* dL_dvdepth, float* dL_dfintense, void* workspace, size_t workspace_bytes,
                             bool deterministic, dmr_stream_t stream_, float* dL_dmv = nullptr, float* dL_dproj = nullptr,
                             bool exact = false, const float* dL_dalpha = nullptr)
{
    const bool cam = dL_dmv != nullptr;
    cudaStream_t stream = (cudaStream_t)stream_;
    if (!sizes_ok(B, P, F, W, H) || R < 0) return DMR_ETOOLARGE;
    if (B == 0 || F == 0 || R == 0) return DMR_OK;   // nothing was composited: all gradients stay zero
    if (!background || !inv_mv_mats || !inv_proj_mats || !face_buffer || !binning_buffer || !image_buffer ||
        !dL_dcolor || !dL_ddepth || !dL_dverts || !dL_dvcolor || !dL_dfopacity || !dL_dvdepth || !dL_dfintense) {
        set_error("null pointer");
        return DMR_EINVAL;
    }
    (void)point_buffer;
    TriFaceLayout FL = TriFaceLayout::make((size_t)B * F);
    TriImageLayout IL = TriImageLayout::make(B, W, H);
    BinningLayout BL = BinningLayout::make((size_t)R);
    TriRenderParams p = {};
    p.B = B; p.F = F; p.W = W; p.H = H; p.P = P;
    p.ranges = at<uint2>(image_buffer, IL.ranges);
    p.face_list = at<uint32_t>(binning_buffer, BL.vals_sorted);
    p.records = at<TriRecord>(face_buffer, FL.records);
    p.bg = background; p.inv_mv = inv_mv_mats; p.inv_proj = inv_proj_mats;
    p.final_T = const_cast<float*>(at<float>(image_buffer, IL.final_T));
    p.prev_T = const_cast<float*>(at<float>(image_buffer, IL.prev_T));
    p.n_contrib = const_cast<uint32_t*>(at<uint32_t>(image_buffer, IL.n_contrib));
    p.dL_dcolor = dL_dcolor; p.dL_ddepth = dL_ddepth;
    p.dL_dverts = dL_dverts; p.dL_dvcolor = dL_dvcolor; p.dL_dfopacity = dL_dfopacity;
    p.dL_dvdepth = dL_dvdepth; p.dL_dfintense = dL_dfintense;
    // camera gradients: one 96-byte record per (view, tile) behind the mode's own scratch, written by every CTA
    // (empty tiles store zeros), so it is not cleared
    const size_t base_bytes = deterministic ? TriDetLayout::make((size_t)B, (size_t)P, (size_t)F).total
                                            : TriBwdLayout::make((size_t)B * F, (size_t)P).total;
    float* cam_tiles = nullptr;
    if (cam) {
        const size_t need = tri_cam_bytes(B, P, F, W, H, deterministic);
        if (!workspace || workspace_bytes < need) {
            set_error("camera-gradient backward needs a workspace of %zu bytes (dmr_tri_backward_camera_bytes)", need);
            return DMR_EINVAL;
        }
        cam_tiles = at<float>(workspace, align_up(base_bytes, 256));
    }
    if (deterministic) {
        TriDetLayout DL = TriDetLayout::make((size_t)B, (size_t)P, (size_t)F);
        void* det_workspace = workspace;
        if (!det_workspace || workspace_bytes < DL.total) {
            set_error("deterministic backward needs a workspace of %zu bytes (dmr_tri_backward_deterministic_bytes)", DL.total);
            return DMR_EINVAL;
        }
        p.det_gmax = at<uint32_t>(det_workspace, DL.gmax);
        p.det_stats = at<long long>(det_workspace, DL.stats);
        p.det_vert = at<long long>(det_workspace, DL.vert);
        p.det_vdepth = at<long long>(det_workspace, DL.vdepth);
        p.det_fopa = at<long long>(det_workspace, DL.fopa);
        DMR_CUDA(cudaMemsetAsync(det_workspace, 0, DL.total, stream));
        int rc = tri_render_backward_deterministic(p, stream, cam_tiles, exact, dL_dalpha);
        if (rc || !cam) return rc;
        return tri_camera_finish(B, W, H, cam_tiles, inv_mv_mats, inv_proj_mats, dL_dmv, dL_dproj, stream);
    }
    // backward scratch: the caller's workspace (the forward's state buffers stay read-only)
    TriBwdLayout WL = TriBwdLayout::make((size_t)B * F, (size_t)P);
    if (!workspace || workspace_bytes < WL.total) {
        set_error("backward needs a workspace of %zu bytes (dmr_tri_backward_workspace_bytes)", WL.total);
        return DMR_EINVAL;
    }
    p.grad_stats = at<float>(workspace, WL.grad_stats);
    // per-vertex vector accumulators only when the vertices are shared (the finish kernel scatters once per FACE, the
    // views already summed: 3F vertex references; from ~4 references per vertex two vector reductions + the fold
    // kernel beat six scalar atomics per reference)
    const bool use_vacc = 3 * (size_t)F >= 4 * (size_t)P;
    p.grad_vacc = use_vacc ? at<float4>(workspace, WL.grad_vacc) : nullptr;
    DMR_CUDA(cudaMemsetAsync(workspace, 0, use_vacc ? WL.total - 256 : WL.stats_end, stream));
    int rc = tri_render_backward(p, stream, cam_tiles, exact, dL_dalpha);
    if (rc || !cam) return rc;
    return tri_camera_finish(B, W, H, cam_tiles, inv_mv_mats, inv_proj_mats, dL_dmv, dL_dproj, stream);
}

int dmr_tri_backward(int B, int P, int F, int W, int H, int R, const float* background, const float* inv_mv_mats,
                     const float* inv_proj_mats, const void* point_buffer, const void* face_buffer,
                     const void* binning_buffer, const void* image_buffer, const float* dL_dcolor,
                     const float* dL_ddepth, float* dL_dverts, float* dL_dvcolor, float* dL_dfopacity,
                     float* dL_dvdepth, float* dL_dfintense, void* workspace, size_t workspace_bytes, dmr_stream_t stream)
{
    return tri_backward_impl(B, P, F, W, H, R, background, inv_mv_mats, inv_proj_mats, point_buffer, face_buffer,
                             binning_buffer, image_buffer, dL_dcolor, dL_ddepth, dL_dverts, dL_dvcolor, dL_dfopacity,
                             dL_dvdepth, dL_dfintense, workspace, workspace_bytes, false, stream);
}

size_t dmr_tri_backward_workspace_bytes(int B, int P, int F)
{
    if (B < 0 || P < 0 || F < 0) return 0;
    return TriBwdLayout::make((size_t)B * F, (size_t)P).total;
}

size_t dmr_tri_backward_deterministic_bytes(int B, int P, int F)
{
    if (B < 0 || P < 0 || F < 0) return 0;
    return TriDetLayout::make((size_t)B, (size_t)P, (size_t)F).total;
}

int dmr_tri_backward_deterministic(int B, int P, int F, int W, int H, int R, const float* background,
                                   const float* inv_mv_mats, const float* inv_proj_mats, const void* point_buffer,
                                   const void* face_buffer, const void* binning_buffer, const void* image_buffer,
                                   const float* dL_dcolor, const float* dL_ddepth, float* dL_dverts, float* dL_dvcolor,
                                   float* dL_dfopacity, float* dL_dvdepth, float* dL_dfintense, void* workspace,
                                   size_t workspace_bytes, dmr_stream_t stream)
{
    return tri_backward_impl(B, P, F, W, H, R, background, inv_mv_mats, inv_proj_mats, point_buffer, face_buffer,
                             binning_buffer, image_buffer, dL_dcolor, dL_ddepth, dL_dverts, dL_dvcolor, dL_dfopacity,
                             dL_dvdepth, dL_dfintense, workspace, workspace_bytes, true, stream);
}

size_t dmr_tri_backward_camera_bytes(int B, int P, int F, int W, int H, int deterministic)
{
    if (B < 0 || P < 0 || F < 0 || W < 0 || H < 0) return 0;
    return tri_cam_bytes(B, P, F, W, H, deterministic != 0);
}

int dmr_tri_backward_camera(int B, int P, int F, int W, int H, int R, const float* background, const float* inv_mv_mats,
                            const float* inv_proj_mats, const void* point_buffer, const void* face_buffer,
                            const void* binning_buffer, const void* image_buffer, const float* dL_dcolor,
                            const float* dL_ddepth, float* dL_dverts, float* dL_dvcolor, float* dL_dfopacity,
                            float* dL_dvdepth, float* dL_dfintense, int deterministic, float* dL_dmv, float* dL_dproj,
                            void* workspace, size_t workspace_bytes, dmr_stream_t stream)
{
    if (B > 0 && (!dL_dmv || !dL_dproj)) { set_error("null pointer"); return DMR_EINVAL; }
    return tri_backward_impl(B, P, F, W, H, R, background, inv_mv_mats, inv_proj_mats, point_buffer, face_buffer,
                             binning_buffer, image_buffer, dL_dcolor, dL_ddepth, dL_dverts, dL_dvcolor, dL_dfopacity,
                             dL_dvdepth, dL_dfintense, workspace, workspace_bytes, deterministic != 0, stream, dL_dmv,
                             dL_dproj);
}

int dmr_tri_backward_exact(int B, int P, int F, int W, int H, int R, const float* background, const float* inv_mv_mats,
                           const float* inv_proj_mats, const void* point_buffer, const void* face_buffer,
                           const void* binning_buffer, const void* image_buffer, const float* dL_dcolor,
                           const float* dL_ddepth, float* dL_dverts, float* dL_dvcolor, float* dL_dfopacity,
                           float* dL_dvdepth, float* dL_dfintense, int deterministic, float* dL_dmv, float* dL_dproj,
                           void* workspace, size_t workspace_bytes, dmr_stream_t stream)
{
    if ((dL_dmv == nullptr) != (dL_dproj == nullptr)) { set_error("pass both dL_dmv and dL_dproj, or neither"); return DMR_EINVAL; }
    return tri_backward_impl(B, P, F, W, H, R, background, inv_mv_mats, inv_proj_mats, point_buffer, face_buffer,
                             binning_buffer, image_buffer, dL_dcolor, dL_ddepth, dL_dverts, dL_dvcolor, dL_dfopacity,
                             dL_dvdepth, dL_dfintense, workspace, workspace_bytes, deterministic != 0, stream, dL_dmv,
                             dL_dproj, true);
}

int dmr_tri_backward_alpha(int B, int P, int F, int W, int H, int R, const float* background, const float* inv_mv_mats,
                           const float* inv_proj_mats, const void* point_buffer, const void* face_buffer,
                           const void* binning_buffer, const void* image_buffer, const float* dL_dcolor,
                           const float* dL_ddepth, float* dL_dverts, float* dL_dvcolor, float* dL_dfopacity,
                           float* dL_dvdepth, float* dL_dfintense, int deterministic, int exact, float* dL_dmv,
                           float* dL_dproj, const float* dL_dalpha, void* workspace, size_t workspace_bytes,
                           dmr_stream_t stream)
{
    if ((dL_dmv == nullptr) != (dL_dproj == nullptr)) { set_error("pass both dL_dmv and dL_dproj, or neither"); return DMR_EINVAL; }
    if (B > 0 && !dL_dalpha) { set_error("null pointer: dL_dalpha"); return DMR_EINVAL; }
    return tri_backward_impl(B, P, F, W, H, R, background, inv_mv_mats, inv_proj_mats, point_buffer, face_buffer,
                             binning_buffer, image_buffer, dL_dcolor, dL_ddepth, dL_dverts, dL_dvcolor, dL_dfopacity,
                             dL_dvdepth, dL_dfintense, workspace, workspace_bytes, deterministic != 0, stream, dL_dmv,
                             dL_dproj, exact != 0, dL_dalpha);
}

int dmr_tri_alpha(int B, int W, int H, const void* image_buffer, float* out_alpha, dmr_stream_t stream)
{
    if (!sizes_ok(B, 0, 0, W, H)) return DMR_ETOOLARGE;
    if (B == 0) return DMR_OK;
    if (!image_buffer || !out_alpha) { set_error("null pointer"); return DMR_EINVAL; }
    const TriImageLayout IL = TriImageLayout::make(B, W, H);
    return image_alpha(false, B, W, H, at<float>(image_buffer, IL.final_T), nullptr, out_alpha, (cudaStream_t)stream);
}

size_t dmr_tri_background_grad_bytes(int B) { return B < 0 ? 0 : image_bg_grad_bytes(B); }

int dmr_tri_background_grad(int B, int W, int H, const void* image_buffer, const float* dL_dcolor, float* dL_dbg,
                            void* workspace, size_t workspace_bytes, dmr_stream_t stream)
{
    if (!sizes_ok(B, 0, 0, W, H)) return DMR_ETOOLARGE;
    if (!dL_dbg) { set_error("null pointer: dL_dbg"); return DMR_EINVAL; }
    if (B > 0 && (!image_buffer || !dL_dcolor)) { set_error("null pointer"); return DMR_EINVAL; }
    const size_t need = image_bg_grad_bytes(B);
    if (!workspace || workspace_bytes < need) {
        set_error("background gradient needs a workspace of %zu bytes (dmr_tri_background_grad_bytes)", need);
        return DMR_EINVAL;
    }
    if (B == 0) { DMR_CUDA(cudaMemsetAsync(dL_dbg, 0, 3 * sizeof(float), (cudaStream_t)stream)); return DMR_OK; }
    const TriImageLayout IL = TriImageLayout::make(B, W, H);
    return image_bg_grad(false, B, W, H, at<float>(image_buffer, IL.final_T), nullptr, dL_dcolor, dL_dbg, workspace,
                         (cudaStream_t)stream);
}

size_t dmr_tri_depth_chain_camera_bytes(int B, int P)
{
    if (B < 0 || P < 0) return 0;
    return depth_chain_camera_bytes(B, P);
}

int dmr_tri_depth_chain_camera(int B, int P, const float* verts, const float* mv_mats, const float* proj_mats,
                               const float* dL_dvdepth, float* dL_dverts, float* dL_dmv, float* dL_dproj, void* workspace,
                               size_t workspace_bytes, dmr_stream_t stream)
{
    if (B < 0 || P < 0) { set_error("negative size"); return DMR_EINVAL; }
    if (B == 0 || P == 0) return DMR_OK;
    if (!verts || !mv_mats || !proj_mats || !dL_dvdepth || !dL_dverts || !dL_dmv || !dL_dproj) {
        set_error("null pointer");
        return DMR_EINVAL;
    }
    const size_t need = depth_chain_camera_bytes(B, P);
    if (!workspace || workspace_bytes < need) {
        set_error("camera depth chain needs a workspace of %zu bytes (dmr_tri_depth_chain_camera_bytes)", need);
        return DMR_EINVAL;
    }
    int rc = depth_chain(B, P, verts, mv_mats, proj_mats, dL_dvdepth, dL_dverts, (cudaStream_t)stream);
    if (rc) return rc;
    return depth_chain_camera(B, P, verts, mv_mats, proj_mats, dL_dvdepth, dL_dmv, dL_dproj, workspace, (cudaStream_t)stream);
}

int dmr_debug_view(int renderer, int kind, int B, int P, int F, int T, int W, int H, size_t R, const void* buffer,
                   const void** ptr, size_t* count)
{
    if (!buffer || !ptr || !count) { set_error("null pointer"); return DMR_EINVAL; }
    (void)T;
    const size_t BF = (size_t)B * F, BP = (size_t)B * P, BI = (size_t)B * W * H;
    const size_t tiles = (size_t)B * ((W + DMR_TILE - 1) / DMR_TILE) * ((H + DMR_TILE - 1) / DMR_TILE);
    size_t off = 0, n = 0;
    if (kind == DMR_VIEW_VERTS_IMAGE) { off = 0; n = BP; }
    else if (kind >= DMR_VIEW_KEYS_UNSORTED && kind <= DMR_VIEW_VALUES_SORTED) {
        BinningLayout L = BinningLayout::make(R);
        n = R;
        off = kind == DMR_VIEW_KEYS_UNSORTED ? L.keys_unsorted : kind == DMR_VIEW_VALUES_UNSORTED ? L.vals_unsorted
            : kind == DMR_VIEW_KEYS_SORTED ? L.keys_sorted : L.vals_sorted;
    } else if (renderer == 0) {
        TriFaceLayout FL = TriFaceLayout::make(BF);
        TriImageLayout IL = TriImageLayout::make(B, W, H);
        switch (kind) {
        case DMR_VIEW_TILES_TOUCHED: off = FL.bin.tiles_touched; n = BF; break;
        case DMR_VIEW_FACE_OFFSETS:  off = FL.bin.offsets; n = BF; break;
        case DMR_VIEW_DEPTH_KEYS:    off = FL.bin.depth_key; n = BF; break;
        case DMR_VIEW_FACE_ORDER:    off = FL.bin.order; n = BF; break;
        case DMR_VIEW_RANGES:        off = IL.ranges; n = tiles; break;
        case DMR_VIEW_N_CONTRIB:     off = IL.n_contrib; n = BI; break;
        case DMR_VIEW_FINAL_T:       off = IL.final_T; n = BI; break;
        default: set_error("unknown view kind %d", kind); return DMR_EINVAL;
        }
    } else {
        TetFaceLayout FL = TetFaceLayout::make(BF, (size_t)F);
        TetImageLayout IL = TetImageLayout::make(B, W, H);
        switch (kind) {
        case DMR_VIEW_TILES_TOUCHED: off = FL.bin.tiles_touched; n = BF; break;
        case DMR_VIEW_FACE_OFFSETS:  off = FL.bin.offsets; n = BF; break;
        case DMR_VIEW_DEPTH_KEYS:    off = FL.bin.depth_key; n = BF; break;
        case DMR_VIEW_FACE_ORDER:    off = FL.bin.order; n = BF; break;
        case DMR_VIEW_RANGES:        off = IL.ranges; n = tiles; break;
        case DMR_VIEW_N_CONTRIB:     off = IL.n_contrib; n = BI; break;
        case DMR_VIEW_FINAL_T:       off = IL.final_log_T; n = BI; break;
        case DMR_VIEW_FIRST_FACE:    off = IL.first_face; n = BI; break;
        case DMR_VIEW_FIRST_TET:     off = IL.first_tet; n = BI; break;
        case DMR_VIEW_TET_JITTER:    off = IL.jitter; n = BI; break;
        default: set_error("unknown view kind %d", kind); return DMR_EINVAL;
        }
    }
    *ptr = static_cast<const unsigned char*>(buffer) + off;
    *count = n;
    return DMR_OK;
}

}  // extern "C"
