/*
 * dmesh_b200.h -- C ABI of libdmesh_b200.so
 *
 * B200-native (sm_100a) replacement for the hot path of SonSang/dmesh_renderer:
 * the tile-based differentiable rasterizer, tri renderer (cuda_rasterizer/) and
 * tet renderer (cuda_renderer/).  Plain pointers and sizes only; no torch types.
 *
 * Each entry point names the reference interface it replaces (paths relative to
 * the reference repository).  The Python `_C` shim
 * (dmesh_renderer_b200/_C.py) binds exactly these symbols and re-creates the
 * four pybind functions of ext.cpp:4-12 on top of them.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless its name ends in `_host`
 *   - all work is enqueued on `stream` (a cudaStream_t); the library never
 *     synchronises the device except where stated and never allocates device
 *     memory.  Rendering state lives entirely in the caller's buffers (calls on
 *     different streams / threads are independent); the only process-wide state
 *     is diagnostic: the launch counter, the dmr_profile_* stage timers and the
 *     dmr_debug_set_* test hooks (not thread-safe, off by default)
 *   - return value: 0 on success, non-zero DMR_E* code otherwise; the message
 *     is available through dmr_last_error() (thread-local)
 *   - matrices are the 16 floats of the reference's column-major convention
 *     (cuda_rasterizer/auxiliary.h:71-90): x' = m[0]x + m[4]y + m[8]z + m[12]
 *   - tile size is fixed at 16x16 (cuda_rasterizer/config.h:4-6)
 */
#ifndef DMESH_B200_H_
#define DMESH_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DMR_OK            0
#define DMR_EINVAL        1   /* bad argument (null pointer, negative size ...)   */
#define DMR_ECUDA         2   /* a CUDA runtime call or kernel launch failed      */
#define DMR_ETOOLARGE     3   /* a size exceeds the 32-bit index budget of a stage */

typedef void* dmr_stream_t;   /* cudaStream_t */

/* Library identification. */
int         dmr_abi_version(void);
const char* dmr_last_error(void);

/* ------------------------------------------------------------------------ */
/* Sizes of the opaque state buffers.                                        */
/* Replaces required<VertState|FaceState|ImageState>() and the resize        */
/* lambdas: cuda_rasterizer/rasterizer_impl.h:61-67, render.cu:18-24,        */
/* rasterizer_impl.cu:200-221 (tri); cuda_renderer/renderer_impl.cu:225-238. */
/* out[0]=point buffer, out[1]=face buffer, out[2]=image buffer (bytes).     */
/* ------------------------------------------------------------------------ */
int    dmr_tri_state_bytes(int B, int P, int F, int W, int H, size_t out[3]);
int    dmr_tet_state_bytes(int B, int P, int F, int T, int W, int H, size_t out[3]);
/* The tet renderer's view-independent adjacency records (one 128-byte record per tet, replacing the per-step   */
/* gathers of cuda_renderer/forward.cu:672-768).  They depend only on verts / faces / tets / face_tets /         */
/* tet_faces, so a caller may build them once and reuse the buffer for every later call on the same geometry     */
/* (dmr_tet_forward_bin: tet_records_valid).  A caller that optimises verts (dmr_tet_backward_vertex) changes     */
/* that geometry in every step and has to rebuild them after each change.                                         */
size_t dmr_tet_records_bytes(int T);
/* Builds them stand-alone (dmr_tet_forward_bin does the same when tet_records_valid == 0). */
int    dmr_tet_build_records(int P, int F, int T, const float* verts, const int* faces, const int* tets,
                             const int* face_tets, const int* tet_faces, void* tet_records, dmr_stream_t stream);
/* Replaces required<BinningState>(R): rasterizer_impl.cu:297-299.           */
size_t dmr_binning_bytes(size_t R);

/* Host-side wait for the num_rendered read-back of *_forward_bin: the caller  */
/* stores `sentinel` (a value num_rendered cannot take, e.g. INT32_MIN) in the  */
/* pinned word before calling *_forward_bin and waits here until the copy has  */
/* overwritten it.  Replaces the blocking 4-byte cudaMemcpy + device sync of   */
/* rasterizer_impl.cu:287-292 / renderer_impl.cu:305-310 with a spin on the    */
/* pinned word (falls back to cudaStreamSynchronize(stream)).                  */
int dmr_wait_i32(volatile int32_t* host_value, int32_t sentinel, dmr_stream_t stream);

/* ------------------------------------------------------------------------ */
/* inverse(mv_mats), inverse(proj_mats) of B cameras in one launch.          */
/* Replaces the two th.inverse calls of the reference's Python wrapper        */
/* (dmesh_renderer/__init__.py:62-63 tri, 298-299 tet) -- ~24 library kernels  */
/* and two device synchronisations -- with the same LU / triangular-solve      */
/* arithmetic done by one thread per matrix; bit-identical to torch.inverse on */
/* this stack (csrc/inverse.cu).  Inputs are [B,4,4] fp32 with arbitrary       */
/* element strides (the API passes transposed views).  `out`: 4*B*16 floats,   */
/* 16-byte aligned = contiguous [mv | proj | inverse(mv) | inverse(proj)].     */
/* `info`: 2*B int32, device-accessible (device memory or mapped pinned host   */
/* memory): LAPACK getrf info per matrix, > 0 = singular (the caller raises).  */
/* ------------------------------------------------------------------------ */
int dmr_camera_inverses(int B, const float* mv_mats, int64_t mv_batch_stride, int64_t mv_row_stride,
                        int64_t mv_col_stride, const float* proj_mats, int64_t proj_batch_stride,
                        int64_t proj_row_stride, int64_t proj_col_stride, float* out, int32_t* info,
                        dmr_stream_t stream);

/* ------------------------------------------------------------------------ */
/* Tri renderer, forward, phase 1: preprocess + per-face records + scan.     */
/* Replaces stages T1-T4 of CudaRasterizer::Rasterizer::forward              */
/* (cuda_rasterizer/rasterizer_impl.cu:226-292): preprocessPointCUDA         */
/* (forward.cu:17-47), preprocessFaceCUDA (forward.cu:76-149),               */
/* cub::DeviceScan::InclusiveSum and the 4-byte D2H of num_rendered.         */
/* `num_rendered_host` must be pinned host memory; the value is valid after  */
/* the caller synchronises `stream` (this call does not synchronise).        */
/* ------------------------------------------------------------------------ */
int dmr_tri_forward_bin(
    int B, int P, int F, int W, int H,
    const float* verts,          /* [P,3]   */
    const int*   faces,          /* [F,3]   */
    const float* verts_color,    /* [P,3]   */
    const float* faces_opacity,  /* [F]     */
    const float* mv_mats,        /* [B,16]  */
    const float* proj_mats,      /* [B,16]  */
    const float* verts_depth,    /* [B,P] or NULL = fused NDC z */
    const float* faces_intense,  /* [B,F]   */
    void* point_buffer, void* face_buffer,
    int32_t* num_rendered_host,
    dmr_stream_t stream);

/* Fused vertex depth (no reference counterpart; SURVEY.md 8f-1).  With verts_depth == NULL in                  */
/* dmr_tri_forward_bin the per-view vertex depth is the vertex's own NDC z (what DMesh's callers compute         */
/* upstream and pass in as verts_depth[B,P]); dmr_tri_backward still returns dL_dvdepth[B,P] and this call        */
/* adds its chain through the projection to dL_dverts[P,3]:  dL/dp += sum_b dL_dvdepth[b,p] * d ndc_z / dp.       */
int dmr_tri_depth_chain(int B, int P, const float* verts, const float* mv_mats, const float* proj_mats,
                        const float* dL_dvdepth, float* dL_dverts, dmr_stream_t stream);


/* ------------------------------------------------------------------------ */
/* Tri renderer, forward, phase 2: binning + sort + tile ranges + render.    */
/* Replaces stages T5-T10 (rasterizer_impl.cu:297-380): duplicateWithKeys    */
/* (rasterizer_impl.cu:44-97), cub::DeviceRadixSort::SortPairs (319-324),    */
/* the ranges memset + identifyTileRanges (102-124, 330-337),                */
/* generateRaysCUDA (forward.cu:184-231) and renderCUDA (forward.cu:257-489).*/
/* out_color [B,3,H,W], out_depth [B,1,H,W] are fully written.               */
/* `R` = the number of instances `binning_buffer` was sized and is laid out  */
/* for (dmr_binning_bytes(R)): num_rendered itself, or any larger capacity.  */
/* The kernels read the real instance count on the device (the scan's total  */
/* in `face_buffer`), so this call may be enqueued BEFORE num_rendered has   */
/* reached the host.  If the real count exceeds R nothing is emitted (all    */
/* tile ranges empty, background image): call again with a buffer that fits. */
/* Pass the same R to dmr_tri_backward.                                      */
/* ------------------------------------------------------------------------ */
int dmr_tri_forward_render(
    int B, int P, int F, int W, int H, int R,
    const float* background,     /* [3] device */
    const float* inv_mv_mats,    /* [B,16] */
    const float* inv_proj_mats,  /* [B,16] */
    const void* point_buffer, void* face_buffer,
    void* binning_buffer, void* image_buffer,
    float* out_color, float* out_depth,
    dmr_stream_t stream);

/* ------------------------------------------------------------------------ */
/* Tri renderer, backward.                                                   */
/* Replaces CudaRasterizer::Rasterizer::backward                              */
/* (rasterizer_impl.cu:387-467) -> TRI_BACKWARD::renderCUDA                   */
/* (cuda_rasterizer/backward.cu:9-421).  The five gradient buffers must be   */
/* zero-initialised by the caller (the reference does torch::zeros,          */
/* render.cu:166-171); gradients are accumulated into them.  The four state  */
/* buffers of the forward call are only READ (a saved-for-backward tensor is */
/* never modified, so several backward passes of one forward may run         */
/* concurrently); the per-(view, face) gradient statistics and per-vertex    */
/* accumulators live in `workspace`: device scratch of                       */
/* dmr_tri_backward_workspace_bytes(B, P, F) bytes, zeroed by the call, free  */
/* again once the work enqueued by the call has completed.                   */
/* ------------------------------------------------------------------------ */
size_t dmr_tri_backward_workspace_bytes(int B, int P, int F);
int dmr_tri_backward(
    int B, int P, int F, int W, int H, int R,
    const float* background,
    const float* inv_mv_mats, const float* inv_proj_mats,
    const void* point_buffer, const void* face_buffer,
    const void* binning_buffer, const void* image_buffer,
    const float* dL_dcolor,      /* [B,3,H,W] */
    const float* dL_ddepth,      /* [B,1,H,W] */
    float* dL_dverts,            /* [P,3]  summed over views */
    float* dL_dvcolor,           /* [P,3]  summed over views */
    float* dL_dfopacity,         /* [F]    summed over views */
    float* dL_dvdepth,           /* [B,P]  */
    float* dL_dfintense,         /* [B,F]  */
    void* workspace, size_t workspace_bytes,
    dmr_stream_t stream);

/* The same with run-to-run REPRODUCIBLE gradients (SURVEY.md 8f-3; the reference's scalar atomics,             */
/* cuda_rasterizer/backward.cu:389-415, give different low-order bits on every run).  Identical kernels up to     */
/* the accumulation; the partial sums are accumulated as 64-bit fixed-point integers, scaled relative to           */
/* max |dL_dout| (integer addition is associative, so the arrival order no longer matters), and converted once.    */
/* Resolution 2^-38 of max |dL_dout| for colour / opacity / intensity / depth terms, 2^-28 for vertex positions;   */
/* results agree with dmr_tri_backward within fp32 accumulation noise.  `workspace`: device scratch of            */
/* dmr_tri_backward_deterministic_bytes(B, P, F) bytes (zeroed by the call).  The gradients are ADDED to the five  */
/* output buffers, as in dmr_tri_backward.                                                                        */
size_t dmr_tri_backward_deterministic_bytes(int B, int P, int F);
int dmr_tri_backward_deterministic(
    int B, int P, int F, int W, int H, int R,
    const float* background,
    const float* inv_mv_mats, const float* inv_proj_mats,
    const void* point_buffer, const void* face_buffer,
    const void* binning_buffer, const void* image_buffer,
    const float* dL_dcolor, const float* dL_ddepth,
    float* dL_dverts, float* dL_dvcolor, float* dL_dfopacity, float* dL_dvdepth, float* dL_dfintense,
    void* workspace, size_t workspace_bytes,
    dmr_stream_t stream);

/* Camera gradients of the tri renderer (no reference counterpart: the reference returns no gradient for the      */
/* matrices).  The same backward pass as dmr_tri_backward (deterministic == 0) or dmr_tri_backward_deterministic  */
/* (deterministic != 0), with the same arguments and the same five gradients, plus dL/dmv_mats and                */
/* dL/dproj_mats [B,16] (column-major, like the matrices), ADDED to the caller's zeroed buffers.  The derivative   */
/* is that of the rays (ray origin and direction formed from inv_mv_mats / inv_proj_mats) with coverage, depth    */
/* order and n_contrib held fixed, chained through the inverses (dL/dA = -A^-T dL/dA^-1 A^-T); with the fused     */
/* vertex depth add dmr_tri_depth_chain_camera.  Accumulated without float atomics: reproducible in both modes.  */
/* `workspace`: dmr_tri_backward_camera_bytes(B, P, F, W, H, deterministic) bytes of device scratch.              */
size_t dmr_tri_backward_camera_bytes(int B, int P, int F, int W, int H, int deterministic);
int dmr_tri_backward_camera(
    int B, int P, int F, int W, int H, int R,
    const float* background,
    const float* inv_mv_mats, const float* inv_proj_mats,
    const void* point_buffer, const void* face_buffer,
    const void* binning_buffer, const void* image_buffer,
    const float* dL_dcolor, const float* dL_ddepth,
    float* dL_dverts, float* dL_dvcolor, float* dL_dfopacity, float* dL_dvdepth, float* dL_dfintense,
    int deterministic,
    float* dL_dmv,               /* [B,16] */
    float* dL_dproj,             /* [B,16] */
    void* workspace, size_t workspace_bytes,
    dmr_stream_t stream);

/* Exact vertex-position gradients (no reference counterpart).  The reference's dL_dverts                        */
/* (ray_tri_intersection_grad, auxiliary.h:288-333) differentiates the ray parameter t where the forward pass     */
/* uses the second barycentric v; this entry point differentiates v, so dL_dverts is the derivative of the        */
/* rendered image (coverage, depth order, n_contrib and the clamp region held fixed) and, with camera gradients,  */
/* consistent with dL_dmv / dL_dproj (a rigid motion of scene and camera together changes nothing).  The other    */
/* four gradients and the camera gradients are those of dmr_tri_backward_camera.  Arguments as                    */
/* dmr_tri_backward_camera, except that dL_dmv and dL_dproj may both be NULL (no camera gradients; passing only  */
/* one of them is an error).  `workspace`: the byte count of the mode it modifies --                              */
/* dmr_tri_backward_workspace_bytes, dmr_tri_backward_deterministic_bytes (deterministic != 0) or, with camera    */
/* gradients, dmr_tri_backward_camera_bytes.  Same launches as that mode.                                         */
int dmr_tri_backward_exact(
    int B, int P, int F, int W, int H, int R,
    const float* background,
    const float* inv_mv_mats, const float* inv_proj_mats,
    const void* point_buffer, const void* face_buffer,
    const void* binning_buffer, const void* image_buffer,
    const float* dL_dcolor, const float* dL_ddepth,
    float* dL_dverts, float* dL_dvcolor, float* dL_dfopacity, float* dL_dvdepth, float* dL_dfintense,
    int deterministic,
    float* dL_dmv,               /* [B,16] or NULL */
    float* dL_dproj,             /* [B,16] or NULL */
    void* workspace, size_t workspace_bytes,
    dmr_stream_t stream);

/* Alpha (coverage) cotangent of the tri renderer (no reference counterpart).  The backward pass of               */
/* dmr_tri_backward_exact (exact != 0) or of the reference formula (exact == 0), with the same arguments, plus      */
/* dL_dalpha [B,H,W], the cotangent of alpha = 1 - final_T (dmr_tri_alpha).  alpha depends on the opacities only, so */
/* only dL_dfopacity changes: dL_dalpha enters where the background term does (the per-pixel constant              */
/* bg . dL_dC + dL_dD becomes bg . dL_dC + dL_dD - dL_dalpha).  In deterministic mode the fixed-point scale covers   */
/* max |dL_dalpha| as well.  `workspace`: the byte count of the mode it modifies, as for dmr_tri_backward_exact.     */
/* dL_dalpha must not be NULL for B > 0.                                                                            */
int dmr_tri_backward_alpha(
    int B, int P, int F, int W, int H, int R,
    const float* background,
    const float* inv_mv_mats, const float* inv_proj_mats,
    const void* point_buffer, const void* face_buffer,
    const void* binning_buffer, const void* image_buffer,
    const float* dL_dcolor, const float* dL_ddepth,
    float* dL_dverts, float* dL_dvcolor, float* dL_dfopacity, float* dL_dvdepth, float* dL_dfintense,
    int deterministic, int exact,
    float* dL_dmv,               /* [B,16] or NULL */
    float* dL_dproj,             /* [B,16] or NULL */
    const float* dL_dalpha,      /* [B,H,W] */
    void* workspace, size_t workspace_bytes,
    dmr_stream_t stream);

/* Alpha image of a tri forward call (no reference counterpart): out_alpha[B,H,W] = 1 - final_T, the transmittance */
/* the forward pass multiplied the background by (the T < 1e-4 termination included, so a fully covered pixel gets  */
/* alpha just below 1).  Reads the image buffer of dmr_tri_forward_render; call it after the last phase 2.  With    */
/* R == 0 the image buffer holds final_T = 1 and alpha is 0.                                                         */
int dmr_tri_alpha(int B, int W, int H, const void* image_buffer, float* out_alpha, dmr_stream_t stream);

/* Gradient with respect to the background colour (no reference counterpart): dL_dbg[c] = sum over views and pixels */
/* of final_T * dL_dcolor[b,c,:,:], WRITTEN (not added) to dL_dbg[3].  A fixed-order reduction without float        */
/* atomics (reproducible).  Reads only the image buffer and dL_dcolor, so it applies when R == 0 too.  `workspace`:  */
/* dmr_tri_background_grad_bytes(B) bytes of device scratch.                                                         */
size_t dmr_tri_background_grad_bytes(int B);
int dmr_tri_background_grad(int B, int W, int H, const void* image_buffer, const float* dL_dcolor, float* dL_dbg,
                            void* workspace, size_t workspace_bytes, dmr_stream_t stream);

/* dmr_tri_depth_chain plus the camera part of the fused vertex depth (no reference counterpart):                 */
/* dL_dmv[b] / dL_dproj[b] += sum_p dL_dvdepth[b,p] * d ndc_z[b,p] / d(mv_mats[b], proj_mats[b]) (no derivative   */
/* through a clamped clip w).  Reduced in a fixed order without float atomics.  `workspace`:                      */
/* dmr_tri_depth_chain_camera_bytes(B, P) bytes of device scratch.                                                */
size_t dmr_tri_depth_chain_camera_bytes(int B, int P);
int dmr_tri_depth_chain_camera(int B, int P, const float* verts, const float* mv_mats, const float* proj_mats,
                               const float* dL_dvdepth, float* dL_dverts, float* dL_dmv, float* dL_dproj,
                               void* workspace, size_t workspace_bytes, dmr_stream_t stream);

/* ------------------------------------------------------------------------ */
/* Tet renderer, forward, phase 1.  Replaces E1, E4, E5 of                   */
/* CudaRenderer::Renderer::forward (cuda_renderer/renderer_impl.cu:241-310): */
/* preprocessPointCUDA (cuda_renderer/forward.cu:21-52), preprocessFaceCUDA  */
/* (178-260), InclusiveSum + D2H; and builds the per-tet adjacency records   */
/* that replace the per-step gathers of cuda_renderer/forward.cu:672-768.    */
/* ------------------------------------------------------------------------ */
int dmr_tet_forward_bin(
    int B, int P, int F, int T, int W, int H,
    const float* verts, const int* faces,
    const float* verts_color, const float* faces_opacity,
    const float* mv_mats, const float* proj_mats,
    const int* tets,             /* [T,4] */
    const int* face_tets,        /* [F,2], -1 = none */
    const int* tet_faces,        /* [T,4] */
    void* point_buffer, void* face_buffer,
    void* tet_records,           /* dmr_tet_records_bytes(T) bytes */
    int tet_records_valid,       /* 0: build the records; 1: `tet_records` already holds them for exactly this geometry */
    int32_t* num_rendered_host,
    dmr_stream_t stream);

/* ------------------------------------------------------------------------ */
/* Tet renderer, forward, phase 2.  Replaces E2/E3, E6-E10                   */
/* (renderer_impl.cu:254-262, 312-409): generateRaysCUDA                     */
/* (cuda_renderer/forward.cu:82-145, incl. the cuRAND XORWOW jitter when     */
/* ray_random_seed > 0), duplicateWithKeys on min_depth                      */
/* (renderer_impl.cu:44-99,318-329), SortPairs, identifyTileRanges,          */
/* firstIntersectCUDA (forward.cu:298-445) and the ray-marching renderCUDA   */
/* (forward.cu:485-815).  out_active [B,H,W] is 1.0f / 0.0f.                 */
/* ------------------------------------------------------------------------ */
int dmr_tet_forward_render(
    int B, int P, int F, int T, int W, int H, int R,
    int ray_random_seed,
    const float* background,
    const float* mv_mats, const float* proj_mats,
    const float* inv_mv_mats, const float* inv_proj_mats,
    const float* faces_intense,  /* [B,F] */
    const void* point_buffer, void* face_buffer,
    const void* tet_records,
    void* binning_buffer, void* image_buffer,
    float* out_color, float* out_depth, float* out_active,
    dmr_stream_t stream);

/* dmr_tet_forward_render for views first_view .. first_view + B - 1 of a    */
/* larger job (a camera-sharded multi-view step): the jitter of pixel (x, y) */
/* of call view b uses cuRAND subsequence (first_view + b)*H*W + y*W + x, so */
/* a view gets the same rays whichever call renders it.  first_view = 0 is   */
/* dmr_tet_forward_render; a negative first_view returns DMR_EINVAL before   */
/* any CUDA call.  The backward entry points re-read the stored rays and     */
/* take no first_view.                                                       */
int dmr_tet_forward_render_views(
    int B, int P, int F, int T, int W, int H, int R,
    int ray_random_seed, int first_view,
    const float* background,
    const float* mv_mats, const float* proj_mats,
    const float* inv_mv_mats, const float* inv_proj_mats,
    const float* faces_intense,
    const void* point_buffer, void* face_buffer,
    const void* tet_records,
    void* binning_buffer, void* image_buffer,
    float* out_color, float* out_depth, float* out_active,
    dmr_stream_t stream);

/* ------------------------------------------------------------------------ */
/* Tet renderer, backward.  Replaces CudaRenderer::Renderer::backward        */
/* (renderer_impl.cu:413-498) -> TET_BACKWARD::renderCUDA                    */
/* (cuda_renderer/backward.cu:86-487).  Gradient buffers zeroed by caller.   */
/* The forward call's state buffers are only read; `workspace`: device       */
/* scratch of dmr_tet_backward_workspace_bytes(P) bytes, zeroed by the call. */
/* ------------------------------------------------------------------------ */
size_t dmr_tet_backward_workspace_bytes(int P);
int dmr_tet_backward(
    int B, int P, int F, int T, int W, int H,
    int ray_random_seed,         /* same value as in the forward call */
    const float* background,
    const float* mv_mats, const float* proj_mats,
    const float* inv_mv_mats, const float* inv_proj_mats,
    const float* faces_intense,
    const void* point_buffer, const void* face_buffer,
    const void* tet_records,
    const void* image_buffer,
    const float* dL_dcolor, const float* dL_ddepth,
    float* dL_dverts_color,      /* [P,3] */
    float* dL_dfaces_opacity,    /* [F]   */
    void* workspace, size_t workspace_bytes,
    dmr_stream_t stream);
/* The same with run-to-run reproducible gradients (see dmr_tri_backward_deterministic: the reference's 10 scalar */
/* atomics per crossed face, cuda_renderer/backward.cu:341-360, become two-word fixed-point additions with 48     */
/* fractional bits below max |dL_dout|, 40 for positions).  `workspace`: dmr_tet_backward_deterministic_bytes(P,  */
/* F) bytes of device scratch (zeroed by the call).                                                                */
size_t dmr_tet_backward_deterministic_bytes(int P, int F);
int dmr_tet_backward_deterministic(
    int B, int P, int F, int T, int W, int H,
    int ray_random_seed,
    const float* background,
    const float* mv_mats, const float* proj_mats,
    const float* inv_mv_mats, const float* inv_proj_mats,
    const float* faces_intense,
    const void* point_buffer, const void* face_buffer,
    const void* tet_records,
    const void* image_buffer,
    const float* dL_dcolor, const float* dL_ddepth,
    float* dL_dverts_color, float* dL_dfaces_opacity,
    void* workspace, size_t workspace_bytes,
    dmr_stream_t stream);

/* Camera gradients of the tet renderer (no reference counterpart: the reference returns no gradient for the      */
/* matrices).  The same backward pass as dmr_tet_backward (deterministic == 0) or dmr_tet_backward_deterministic  */
/* (deterministic != 0), with the same arguments and the same two gradients, plus dL/dmv_mats and dL/dproj_mats   */
/* [B,16] (column-major, like the matrices), ADDED to the caller's zeroed buffers.  The derivative is that of the  */
/* forward pass as implemented, with the marched path (first face and tet, faces crossed), n_contrib, termination */
/* and the active mask held fixed, and the branch regions of the clip-w clamp and of the ray-length clamp; it     */
/* flows through the rays (ray origin and direction formed from inv_mv_mats / inv_proj_mats, chained through the  */
/* inverses) and through the hit-point depth (directly through mv_mats / proj_mats).  Only the steps the backward */
/* pass walks contribute (where the reference's reverse march gives up on a ray, its earlier faces get nothing, as */
/* for colour and opacity).  Jittered pixel coordinates (ray_random_seed > 0) are constants.  Accumulated without  */
/* float atomics: reproducible in both modes.  `workspace`: dmr_tet_backward_camera_bytes(B, P, F, W, H,          */
/* deterministic) bytes of device scratch.                                                                         */
size_t dmr_tet_backward_camera_bytes(int B, int P, int F, int W, int H, int deterministic);
int dmr_tet_backward_camera(
    int B, int P, int F, int T, int W, int H,
    int ray_random_seed,
    const float* background,
    const float* mv_mats, const float* proj_mats,
    const float* inv_mv_mats, const float* inv_proj_mats,
    const float* faces_intense,
    const void* point_buffer, const void* face_buffer,
    const void* tet_records,
    const void* image_buffer,
    const float* dL_dcolor, const float* dL_ddepth,
    float* dL_dverts_color, float* dL_dfaces_opacity,
    int deterministic,
    float* dL_dmv,               /* [B,16] */
    float* dL_dproj,             /* [B,16] */
    void* workspace, size_t workspace_bytes,
    dmr_stream_t stream);

/* Vertex-position gradients of the tet renderer (no reference counterpart: the reference returns no gradient for */
/* verts).  The backward pass of dmr_tet_backward_camera, with the same arguments, except that dL_dmv and          */
/* dL_dproj may both be NULL (no camera gradients; passing only one of them is an error), plus dL/dverts [P,3]     */
/* ADDED to dL_dverts.  The derivative is that of the rendered colour and depth images as implemented, with the    */
/* same things held fixed as for the camera gradients; a vertex enters through the (t, u, v) of every walked step  */
/* whose face's triangle (faces[] order) it belongs to.  Only the steps the backward pass walks contribute.  Summed */
/* with float atomics (deterministic == 0) or in fixed point (deterministic != 0; reproducible, NaN for non-finite */
/* cotangents).  The other gradients are those of the mode it extends.  `workspace`:                              */
/* dmr_tet_backward_vertex_bytes(B, P, F, W, H, deterministic, camera) bytes of device scratch, camera = whether  */
/* dL_dmv / dL_dproj are passed: the mode's own scratch plus one per-vertex accumulator.                          */
size_t dmr_tet_backward_vertex_bytes(int B, int P, int F, int W, int H, int deterministic, int camera);
int dmr_tet_backward_vertex(
    int B, int P, int F, int T, int W, int H,
    int ray_random_seed,
    const float* background,
    const float* mv_mats, const float* proj_mats,
    const float* inv_mv_mats, const float* inv_proj_mats,
    const float* faces_intense,
    const void* point_buffer, const void* face_buffer,
    const void* tet_records,
    const void* image_buffer,
    const float* dL_dcolor, const float* dL_ddepth,
    float* dL_dverts_color, float* dL_dfaces_opacity,
    int deterministic,
    float* dL_dmv,               /* [B,16] or NULL */
    float* dL_dproj,             /* [B,16] or NULL */
    float* dL_dverts,            /* [P,3] */
    void* workspace, size_t workspace_bytes,
    dmr_stream_t stream);

/* Face-intensity gradients of the tet renderer (no reference counterpart: the reference returns no gradient for   */
/* faces_intense).  The backward pass of dmr_tet_backward_vertex, with the same arguments, except that dL_dverts   */
/* may be NULL too (no vertex-position gradients), plus dL/dfaces_intense [B,F] ADDED to dL_dfaces_intense.  The    */
/* derivative is that of the rendered colour image (depth does not depend on intensity), with the same things held */
/* fixed as for the camera gradients: per walked step, sum_ch dL/dcol[ch] T alpha interp[ch], interp = the step's   */
/* interpolated vertex colour before the multiplication by the intensity, so a face of intensity 0 gets its        */
/* gradient too.  Only the steps the backward pass walks contribute.  Summed with float atomics (deterministic ==   */
/* 0) or in fixed point (deterministic != 0; reproducible, NaN for non-finite cotangents).  The other gradients are */
/* those of the mode it extends.  `workspace`: dmr_tet_backward_intensity_bytes(B, P, F, W, H, deterministic,       */
/* camera, vertex) bytes of device scratch, camera / vertex = whether dL_dmv and dL_dproj / dL_dverts are passed:   */
/* the mode's own scratch plus, in deterministic mode, one fixed-point accumulator per (view, face).                */
size_t dmr_tet_backward_intensity_bytes(int B, int P, int F, int W, int H, int deterministic, int camera, int vertex);
int dmr_tet_backward_intensity(
    int B, int P, int F, int T, int W, int H,
    int ray_random_seed,
    const float* background,
    const float* mv_mats, const float* proj_mats,
    const float* inv_mv_mats, const float* inv_proj_mats,
    const float* faces_intense,
    const void* point_buffer, const void* face_buffer,
    const void* tet_records,
    const void* image_buffer,
    const float* dL_dcolor, const float* dL_ddepth,
    float* dL_dverts_color, float* dL_dfaces_opacity,
    int deterministic,
    float* dL_dmv,               /* [B,16] or NULL */
    float* dL_dproj,             /* [B,16] or NULL */
    float* dL_dverts,            /* [P,3] or NULL */
    float* dL_dfaces_intense,    /* [B,F] */
    void* workspace, size_t workspace_bytes,
    dmr_stream_t stream);

/* Alpha (coverage) cotangent of the tet renderer (no reference counterpart).  The backward pass of                 */
/* dmr_tet_backward_intensity, with the same arguments, except that dL_dfaces_intense may be NULL too (no intensity  */
/* gradients), plus dL_dalpha [B,H,W], the cotangent of alpha (dmr_tet_alpha).  Only dL_dfaces_opacity changes: the */
/* cotangent enters where the background term does, summed over the same walked steps as every other gradient.      */
/* In deterministic mode the fixed-point scale covers max |dL_dalpha| as well.  `workspace`: the byte count of the   */
/* mode it modifies (dmr_tet_backward_workspace_bytes, _deterministic_bytes, _camera_bytes, _vertex_bytes or         */
/* _intensity_bytes).  dL_dalpha must not be NULL for B > 0.                                                         */
int dmr_tet_backward_alpha(
    int B, int P, int F, int T, int W, int H,
    int ray_random_seed,
    const float* background,
    const float* mv_mats, const float* proj_mats,
    const float* inv_mv_mats, const float* inv_proj_mats,
    const float* faces_intense,
    const void* point_buffer, const void* face_buffer,
    const void* tet_records,
    const void* image_buffer,
    const float* dL_dcolor, const float* dL_ddepth,
    float* dL_dverts_color, float* dL_dfaces_opacity,
    int deterministic,
    float* dL_dmv,               /* [B,16] or NULL */
    float* dL_dproj,             /* [B,16] or NULL */
    float* dL_dverts,            /* [P,3] or NULL */
    float* dL_dfaces_intense,    /* [B,F] or NULL */
    const float* dL_dalpha,      /* [B,H,W] */
    void* workspace, size_t workspace_bytes,
    dmr_stream_t stream);

/* Alpha image of a tet forward call (no reference counterpart): out_alpha[B,H,W] = 1 - expf(final_log_T) on active */
/* pixels (bit-identical to 1 - the transmittance the forward pass multiplied the background by) and 0 on inactive  */
/* ones (numerical failure, shown as the background).  Reads the image buffer of dmr_tet_forward_render(_views).    */
int dmr_tet_alpha(int B, int W, int H, const void* image_buffer, float* out_alpha, dmr_stream_t stream);

/* Gradient with respect to the background colour (no reference counterpart): dL_dbg[c] = sum over views and pixels */
/* of w * dL_dcolor[b,c,:,:], w = expf(final_log_T) on active pixels and 1 on inactive ones, WRITTEN to dL_dbg[3].   */
/* Fixed-order reduction without float atomics.  `workspace`: dmr_tet_background_grad_bytes(B) bytes.               */
size_t dmr_tet_background_grad_bytes(int B);
int dmr_tet_background_grad(int B, int W, int H, const void* image_buffer, const float* dL_dcolor, float* dL_dbg,
                            void* workspace, size_t workspace_bytes, dmr_stream_t stream);

/* ------------------------------------------------------------------------ */
/* Read-only views into the state buffers for the bit-exact parity checks    */
/* (the reference exposes the same quantities through the fromChunk layouts, */
/* rasterizer_impl.cu:127-171).  Returns a device pointer and element count. */
/* ------------------------------------------------------------------------ */
enum dmr_view_kind {
    DMR_VIEW_VERTS_IMAGE    = 0,  /* float4[B*P] {img.x,img.y,ndc.z,depth}   point buffer */
    DMR_VIEW_TILES_TOUCHED  = 1,  /* uint32[B*F]                              face buffer  */
    DMR_VIEW_FACE_OFFSETS   = 2,  /* uint32[B*F] inclusive scan of tiles_touched in FACE_ORDER  face buffer */
    DMR_VIEW_DEPTH_KEYS     = 3,  /* uint32[B*F] float bits of the sort depth face buffer  */
    DMR_VIEW_KEYS_UNSORTED  = 4,  /* uint32[R] tile ids as emitted (depth order)  binning  */
    DMR_VIEW_VALUES_UNSORTED= 5,  /* uint32[R] face ids as emitted               binning   */
    DMR_VIEW_KEYS_SORTED    = 6,  /* uint32[R] tile ids, sorted: the upper word of the      */
                                  /* reference's (tile|depth) key; the lower word is        */
                                  /* DEPTH_KEYS[view*F + value]                  binning   */
    DMR_VIEW_VALUES_SORTED  = 7,  /* uint32[R] face ids in final order           binning   */
    DMR_VIEW_RANGES         = 8,  /* uint2[B*tiles]                           image buffer */
    DMR_VIEW_N_CONTRIB      = 9,  /* uint32[B*W*H]                            image buffer */
    DMR_VIEW_FINAL_T        = 10, /* float[B*W*H] (tet: final log T)          image buffer */
    DMR_VIEW_FIRST_FACE     = 11, /* int32[B*W*H] (tet only)                  image buffer */
    DMR_VIEW_FIRST_TET      = 12, /* int32[B*W*H] (tet only)                  image buffer */
    DMR_VIEW_FACE_ORDER     = 13, /* uint32[B*F] faces (b*F+f) stably sorted by depth key  face buffer */
    DMR_VIEW_TET_JITTER     = 14  /* float2[B*W*H] pixel coordinates of the rays (tet only; written only when */
                                  /* ray_random_seed > 0)                     image buffer */
};
int dmr_debug_view(int renderer /*0=tri,1=tet*/, int kind,
                   int B, int P, int F, int T, int W, int H, size_t R,
                   const void* buffer, const void** ptr, size_t* count);

/* Test hook: number of march steps per ray recorded in the tet renderer's   */
/* face trail (0 = automatic, see tet.cuh).  Changes the image-buffer size   */
/* reported by dmr_tet_state_bytes; set it before the forward call and keep  */
/* it until the matching backward call has been issued.  Not thread-safe.    */
int dmr_debug_set_tet_trail_cap(int cap);
/* Test hook: CTAs per tile of the tet first-intersection search (0 = automatic: 4 up to 4096 tiles,  */
/* 2 up to 16384, else 1).  Results do not depend on it.                                              */
int dmr_debug_set_tet_first_split(int split);

/* ------------------------------------------------------------------------ */
/* Stand-alone stable LSD radix sort of (uint64 key, uint32 value) pairs on  */
/* bits [0, end_bit) -- the hand-written onesweep that replaces              */
/* cub::DeviceRadixSort::SortPairs (rasterizer_impl.cu:319-324).  Exposed    */
/* for unit tests and the sort micro-benchmark.  `temp` must hold            */
/* dmr_sort_temp_bytes(n) bytes.  Inputs are not modified.                   */
/* ------------------------------------------------------------------------ */
size_t dmr_sort_temp_bytes(size_t n);
int    dmr_sort_pairs(const uint64_t* keys_in, const uint32_t* vals_in,
                      uint64_t* keys_out, uint32_t* vals_out,
                      size_t n, int end_bit, void* temp, dmr_stream_t stream);
/* The same sort on 32-bit keys -- the form the renderers use (tile ids of the */
/* instances, depth keys of the faces; two-level binning, DESIGN.md 3.1).      */
/* vals_in == NULL stands for the identity (0, 1, 2, ...).  `temp` as above.   */
int    dmr_sort_pairs_u32(const uint32_t* keys_in, const uint32_t* vals_in,
                          uint32_t* keys_out, uint32_t* vals_out,
                          size_t n, int end_bit, void* temp, dmr_stream_t stream);

/* ------------------------------------------------------------------------ */
/* All-reduce(SUM) of an fp32 buffer that lives in symmetric memory, with the */
/* reduction done inside the NVSwitch (NVLS multimem.ld_reduce / multimem.st).*/
/* No reference counterpart: the reference has no distributed code            */
/* (SURVEY.md 8e); this is the single collective of the camera-sharded step.  */
/* `multicast_ptr` = multicast address of the buffer (every rank passes ITS   */
/* view of the same multicast object), n_floats a multiple of 4*world.  Rank r */
/* reduces and broadcasts slice r, between two cross-GPU barriers inside the  */
/* kernel.  `peer_flag_ptrs_dev`: DEVICE array of `world` pointers, entry r = */
/* rank r's flag words (>= world uint32, zero-initialised symmetric memory);  */
/* `local_ctl`: 2 zero-initialised uint32 on this GPU; `epoch` = 1, 2, 3, ... */
/* (< 2^30) identical on all ranks, one per call on a given flag buffer.      */
/* ------------------------------------------------------------------------ */
int dmr_nvls_allreduce_sum_f32_fused(void* multicast_ptr, size_t n_floats, int rank, int world,
                                     void* const* peer_flag_ptrs_dev, void* local_ctl, unsigned epoch,
                                     dmr_stream_t stream);

/* ------------------------------------------------------------------------ */
/* Per-stage device timing.  No reference counterpart: the reference has no   */
/* tracing at all (SURVEY.md section 5) and serialises every stage with       */
/* cudaDeviceSynchronize (cuda_rasterizer/auxiliary.h:425-432).  When enabled */
/* a pair of CUDA events is recorded on the launching stream around every     */
/* kernel (no synchronisation); dmr_profile_read() waits for the events of    */
/* the most recent call and returns the elapsed milliseconds per stage        */
/* (-1 = stage not run since the last read).  Used by bench.py for the        */
/* roofline of the dominant kernel.  Not thread-safe; one stream at a time.   */
/* ------------------------------------------------------------------------ */
/* Number of kernels this library has launched so far in the process. */
unsigned long long dmr_launch_count(void);
int         dmr_profile_enable(int on);
int         dmr_profile_stage_count(void);
const char* dmr_profile_stage_name(int stage);
int         dmr_profile_read(float* ms_out /* [dmr_profile_stage_count()] */);

#ifdef __cplusplus
}
#endif
#endif /* DMESH_B200_H_ */
