// common.cuh -- shared device helpers, workspace layouts and error plumbing of
// libdmesh_b200.so (sm_100a only).
//
// Numerical contract (SURVEY.md App. A): integer outputs of the binning stages
// must be bit-identical to the reference, so every float expression that feeds
// a float->int conversion keeps the reference's operation order (cited per
// function) and is compiled with nvcc defaults (-fmad=true, IEEE div/sqrt, no
// fast-math), exactly as the reference is built.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stddef.h>

#define DMR_TILE 16            // cuda_rasterizer/config.h:5-6 (BLOCK_X, BLOCK_Y)
#define DMR_T_EPS 0.0001f      // cuda_rasterizer/auxiliary.h:8

namespace dmr {

// ---------------------------------------------------------------------------
// error plumbing
// ---------------------------------------------------------------------------
void set_error(const char* fmt, ...);
int  cuda_fail(cudaError_t e, const char* what);

#define DMR_CUDA(call)                                                     \
    do {                                                                   \
        cudaError_t e__ = (call);                                          \
        if (e__ != cudaSuccess) return ::dmr::cuda_fail(e__, #call);       \
    } while (0)
#define DMR_LAUNCH_CHECK(name)                                             \
    do {                                                                   \
        cudaError_t e__ = cudaGetLastError();                              \
        if (e__ != cudaSuccess) return ::dmr::cuda_fail(e__, name);        \
    } while (0)

// ---------------------------------------------------------------------------
// per-stage timing hook (dmr_profile_*): CUDA events recorded on the launching
// stream around every kernel when enabled; no synchronisation, off by default.
// ---------------------------------------------------------------------------
enum Stage {
    ST_POINTS = 0, ST_FACES, ST_FACE_SORT, ST_SCAN, ST_DUPLICATE, ST_SORT_HIST, ST_SORT_PLAN,
    ST_SORT_PASS0, ST_SORT_PASS1, ST_SORT_PASS2, ST_SORT_PASS3, ST_SORT_PASS4, ST_SORT_PASS5, ST_SORT_PASS6, ST_SORT_PASS7,
    ST_RANGES, ST_TRI_FWD, ST_TRI_BWD, ST_TRI_BWD_FINISH, ST_TET_RECORDS, ST_TET_JITTER, ST_TET_FIRST, ST_TET_FWD, ST_TET_BWD, ST_TET_BWD_FINISH,
    ST_TRI_BWD_CAM, ST_TRI_CAM_FINISH, ST_DEPTH_CAM, ST_DEPTH_CAM_FINISH, ST_TET_BWD_CAM, ST_TET_CAM_FINISH,
    ST_TET_BWD_VERT, ST_TET_BWD_CAM_VERT, ST_TET_VERT_FINISH,
    ST_TET_BWD_INT, ST_TET_BWD_CAM_INT, ST_TET_BWD_VERT_INT, ST_TET_BWD_CAM_VERT_INT, ST_TET_INT_FINISH,
    ST_TRI_ALPHA, ST_TRI_BWD_ALPHA, ST_TRI_BG_GRAD, ST_TET_ALPHA, ST_TET_BWD_ALPHA, ST_TET_BG_GRAD,
    ST_TRI_FACE_WEIGHTS, ST_TET_FACE_WEIGHTS, ST_COUNT
};
void count_launch(int n);
void prof_begin(int stage, cudaStream_t s, bool count = true);   // count: also counts one kernel launch
void prof_end(int stage, cudaStream_t s);
struct ProfScope {
    int st; cudaStream_t s;
    // count = false: a scope around a sequence of launches that count themselves
    ProfScope(int stage, cudaStream_t stream, bool count = true) : st(stage), s(stream) { prof_begin(st, s, count); }
    ~ProfScope() { prof_end(st, s); }
};

// ---------------------------------------------------------------------------
// Programmatic dependent launch (PDL).  A forward call is a chain of 10-15 short kernels on one stream (6-40 us
// each at C1 / C2): with ordinary launches every kernel boundary costs the full launch + drain latency.  Kernels
// launched through dmr_launch carry cudaLaunchAttributeProgrammaticStreamSerialization: the next kernel of the
// chain is set up and its CTAs become resident while the previous one is still draining.  EVERY kernel launched
// this way begins with griddep_wait() -- it blocks until the preceding kernel has completed and its writes are
// visible -- so the data flow is exactly that of ordinary stream order; only the launch latency overlaps.
// ---------------------------------------------------------------------------
__device__ __forceinline__ void griddep_wait()
{
    asm volatile("griddepcontrol.wait;" ::: "memory");
}
template <typename... KArgs, typename... Args>
inline cudaError_t dmr_launch(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Args&&... args)
{
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// ---------------------------------------------------------------------------
// small vector helpers.  dot/cross/transform keep the expression shape of the
// reference (cuda_rasterizer/cuda_math.h:1524-1527, 1696-1699 and
// auxiliary.h:71-90) so that nvcc contracts them into the same FMA chains.
// ---------------------------------------------------------------------------
__device__ __forceinline__ float3 f3(float x, float y, float z) { return make_float3(x, y, z); }
__device__ __forceinline__ float3 operator+(float3 a, float3 b) { return f3(a.x + b.x, a.y + b.y, a.z + b.z); }
__device__ __forceinline__ float3 operator-(float3 a, float3 b) { return f3(a.x - b.x, a.y - b.y, a.z - b.z); }
__device__ __forceinline__ float3 operator-(float3 a) { return f3(-a.x, -a.y, -a.z); }
__device__ __forceinline__ float3 operator*(float3 a, float s) { return f3(a.x * s, a.y * s, a.z * s); }
__device__ __forceinline__ float3 operator*(float s, float3 a) { return f3(s * a.x, s * a.y, s * a.z); }
__device__ __forceinline__ float3 operator*(float3 a, float3 b) { return f3(a.x * b.x, a.y * b.y, a.z * b.z); }
__device__ __forceinline__ float3 operator/(float3 a, float s) { return f3(a.x / s, a.y / s, a.z / s); }
__device__ __forceinline__ float dot3(float3 a, float3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
__device__ __forceinline__ float3 cross3(float3 a, float3 b)
{
    return f3(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x);
}

// Vector reductions (PTX ISA 8.1, sm_90+; SASS REDG.E.ADD.F32x4 / .F32x2).  Measured on B200
// (tools/ubench_red.cu, 47 M scattered 12-float records): 10 scalar reds 2.7-3.3 ms, 3 x v4 0.74-1.7 ms
// -- the LSU/L2 cost of a reduction is per lane-operation, not per float.  No "memory" clobber: the
// kernels that issue them never read the reduced locations, and the clobber would stop the compiler from
// hoisting the next step's loads above a reduction.
__device__ __forceinline__ void red_add_v4(float* a, float x, float y, float z, float w)
{
    asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(a), "f"(x), "f"(y), "f"(z), "f"(w));
}
__device__ __forceinline__ void red_add_v2(float* a, float x, float y)
{
    asm volatile("red.global.add.v2.f32 [%0], {%1, %2};" ::"l"(a), "f"(x), "f"(y));
}

// Per-(view, face) visibility statistics of a forward call (dmr_tri_forward_render_face_weights, dmr_tet_face_weights):
// the sum of the blending weights T * alpha of the face's composited hits as 64-bit fixed point with 32 fractional
// bits (each weight rounded to nearest, so one below 2^-33 adds 0), and the number of those hits.  Integer sums do not
// depend on the order of the reductions: the same bits in every run, without a separate deterministic path.  A weight
// is at most 1 (2^32 in fixed point), so a sum cannot wrap while a view has fewer than 2^31 pixels.
struct FaceWeightAcc {
    unsigned long long* weight;   // [B*F], zeroed
    uint32_t* hits;               // [B*F], zeroed
};
__device__ __forceinline__ void face_weight_add(const FaceWeightAcc& a, size_t i, float w)
{
    const unsigned long long q = __float2ull_rn(w * 4294967296.0f);
    asm volatile("red.global.add.u64 [%0], %1;" ::"l"(a.weight + i), "l"(q));
    asm volatile("red.global.add.u32 [%0], %1;" ::"l"(a.hits + i), "r"(1u));
}

// column-major 4x4 * (p,1): auxiliary.h:71-90
__device__ __forceinline__ float3 xform43(float3 p, const float* m)
{
    return f3(m[0] * p.x + m[4] * p.y + m[8] * p.z + m[12],
              m[1] * p.x + m[5] * p.y + m[9] * p.z + m[13],
              m[2] * p.x + m[6] * p.y + m[10] * p.z + m[14]);
}
__device__ __forceinline__ float4 xform44(float3 p, const float* m)
{
    return make_float4(m[0] * p.x + m[4] * p.y + m[8] * p.z + m[12],
                       m[1] * p.x + m[5] * p.y + m[9] * p.z + m[13],
                       m[2] * p.x + m[6] * p.y + m[10] * p.z + m[14],
                       m[3] * p.x + m[7] * p.y + m[11] * p.z + m[15]);
}

// Entry (i, j) of N^T G N^T for column-major 4x4 N, G (M(r, c) = m[4c + r]).  With N = A^-1 and G = dL/dN, the
// camera-gradient finish kernels of both renderers form dL/dA = -N^T G N^T from it.
__device__ __forceinline__ float inverse_chain(const float* N, const float* G, int i, int j)
{
    float out = 0.0f;
#pragma unroll
    for (int a = 0; a < 4; a++) {
        float h = 0.0f;                                // (G N^T)(a, j) = sum_c G(a, c) N(j, c)
#pragma unroll
        for (int c = 0; c < 4; c++) h += G[4 * c + a] * N[4 * c + j];
        out += N[4 * i + a] * h;                       // N^T(i, a) = N(a, i)
    }
    return out;
}

// auxiliary.h:245-253
__device__ __forceinline__ float clamp_w(float w)
{
    const float eps = 1e-4;
    if (w >= 0 && w < eps) return eps;
    else if (w < 0 && w > -eps) return -eps;
    return w;
}
// auxiliary.h:33-41 -- evaluated in DOUBLE then rounded (App. A.3)
__device__ __forceinline__ float ndc2pix(float v, int S) { return ((v + 1.0) * S - 1.0) * 0.5; }
__device__ __forceinline__ float pix2ndc(float v, int S) { return ((v * 2.0 + 1.0) / S) - 1.0; }

// Pixel ray, tri flavour: cuda_rasterizer/forward.cu:199-230.
// tet flavour (len = max(len,1e-4)): cuda_renderer/forward.cu:129-144.
template <bool TET>
__device__ __forceinline__ void pixel_ray(const float* inv_mv, const float* inv_proj, float pixfx, float pixfy,
                                          int W, int H, float3& ro, float3& rd)
{
    ro = f3(inv_mv[12], inv_mv[13], inv_mv[14]);
    float nx = pix2ndc(pixfx, W);
    float ny = pix2ndc(pixfy, H);
    float4 pv = xform44(f3(nx, ny, -1.0f), inv_proj);
    float4 pw = xform44(f3(pv.x, pv.y, pv.z), inv_mv);
    rd = f3(pw.x, pw.y, pw.z) - ro;
    float len;
    if (TET) {
        len = sqrtf(dot3(rd, rd));
        len = fmaxf(len, 0.0001f);
    } else {
        len = sqrtf(dot3(rd, rd)) + 0.0000001f;
    }
    rd = rd / len;
}

// ---------------------------------------------------------------------------
// raw memory helpers
// ---------------------------------------------------------------------------
__host__ __device__ __forceinline__ size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

__device__ __forceinline__ uint32_t ld_volatile_u32(const uint32_t* p)
{
    uint32_t v;
    asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_volatile_u32(uint32_t* p, uint32_t v)
{
    asm volatile("st.relaxed.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// ---------------------------------------------------------------------------
// Per-(view,face) setup record of the tri renderer: everything the per-tile
// render kernels need, gathered ONCE per face in the face-preprocess kernel so
// that staging an instance is one contiguous 144-byte copy instead of the
// reference's ~10 scattered sectors behind two levels of indirection
// (cuda_rasterizer/forward.cu:358-400).
//
// Edge functions: in_tri() (cuda_rasterizer/auxiliary.h:179-243) evaluates
//     s_k = cx_k*(py - y_k) - cy_k*(px - x_k) - bias_k      (32-bit, wrapping)
// with px = 16*x+8, py = 16*y+8 for the pixel centre.  All operations are ring
// operations mod 2^32, so the affine form
//     s_k = ea[k]*x + eb[k]*y + ec[k]                        (mod 2^32)
// with ea = -16*cy, eb = 16*cx, ec = 8*cx - 8*cy + cy*x_k - cx*y_k - bias is
// bit-identical, including the reference's overflow behaviour.  A degenerate
// triangle (area == 0) is encoded as ea=eb=ec=0 (never covered).
// ---------------------------------------------------------------------------
// (Measured and rejected, round 2: splitting the record in HBM into a 64-byte per-(view, face) part and a 96-byte
// per-face part shared by the views of a call, L2-resident at C4.  The face-preprocess kernel got 27 % faster at 8
// views (383 -> 279 us) and tri_grad_finish 7 %, but staging an instance from two arrays cost the render kernels
// more than that: forward 1842 -> 2033 us, backward 3684 -> 3792 us at C4, forward 420 -> 467 us at C5.)
struct __align__(16) TriRecord {
    // q0..q2: coverage part -- three edge functions; the fourth words carry what no pixel needs
    uint32_t ea0, eb0, ec0; uint32_t flags;   // bit 0: edge values cannot overflow on screen; bits 1..27: block bbox (below)
    uint32_t ea1, eb1, ec1; int i0;           // vertex ids (gradient scatter, tri_grad_finish_kernel); the backward kernel's
    uint32_t ea2, eb2, ec2; int i1;           //   STAGED copy carries the face id in place of i0
    // q3..q8: shading part -- everything a covered pixel reads is exactly these six 16-byte chunks (six LDS.128 per
    // hit; with opacity / intensity in q0 / q1 a hit cost three more scalar loads, and the L1 data pipe is the
    // busiest unit of the render kernels)
    float v0[3]; float opacity;               // world positions
    float v1[3]; float intense;
    float v2[3]; int i2;                      //   the backward kernel's staged copy carries 1 / (1 - opacity) in place of i2
    float c0[3]; float d0;                    // vertex colours, per-view vertex depths
    float c1[3]; float d1;
    float c2[3]; float d2;
};
static_assert(sizeof(TriRecord) == 144, "TriRecord must be 9 x 16 bytes");
#define DMR_REC_WORDS 36
#define DMR_REC_SAFE 1u
// Conservative bounding box of the pixels the (snapped) triangle can cover, in units of the render kernels' warp
// blocks (8 x 4 pixels), packed into `flags`:
//   bits 1..9   first block column (pixel x >> 3)      bits 20..23  number of block columns, 15 = unbounded
//   bits 10..19 first block row    (pixel y >> 2)      bits 24..27  number of block rows,    15 = unbounded
// The three edge-function minima alone keep ~2.5x more instances per block than really touch it (a small triangle
// near a block is rarely separated from it by one of ITS OWN edge lines); the box removes those.  A triangle whose
// box holds no pixel centre at all is stored as degenerate (never covered), which is what in_tri would find.
#define DMR_REC_BX0_SHIFT 1
#define DMR_REC_BY0_SHIFT 10
#define DMR_REC_NBX_SHIFT 20
#define DMR_REC_NBY_SHIFT 24
#define DMR_REC_NB_UNBOUNDED 15u

// ---------------------------------------------------------------------------
// workspace layouts (all offsets 256-byte aligned)
// ---------------------------------------------------------------------------
#define DMR_SCAN_THREADS 256
#define DMR_SCAN_ITEMS 16
#define DMR_SCAN_TILE (DMR_SCAN_THREADS * DMR_SCAN_ITEMS)

size_t sort_temp_bytes_u32(size_t n);

// Per-(view,face) binning scratch at the head of both renderers' face buffers.
//   tiles_touched, depth_key, rect   written by the face-preprocess kernel, indexed by bf = b*F + f
//   order          faces stably sorted by depth key (u32 indices bf)          -- see bin_faces()
//   depth_sorted   the sorted depth keys (sort output, otherwise unused)
//   offsets        inclusive scan of tiles_touched[order[i]]: instance ranges in DEPTH order
struct FaceBinLayout {
    size_t tiles_touched, depth_key, rect, order, depth_sorted, offsets, scan_state, fsort_temp, end;
    __host__ static FaceBinLayout make(size_t BF)
    {
        FaceBinLayout L;
        size_t o = 0;
        L.tiles_touched = o; o = align_up(o + 4 * BF, 256);
        L.depth_key = o;     o = align_up(o + 4 * BF, 256);
        L.rect = o;          o = align_up(o + 8 * BF, 256);
        L.order = o;         o = align_up(o + 4 * BF, 256);
        L.depth_sorted = o;  o = align_up(o + 4 * BF, 256);
        L.offsets = o;       o = align_up(o + 4 * BF, 256);
        size_t ntile = (BF + DMR_SCAN_TILE - 1) / DMR_SCAN_TILE;
        L.scan_state = o;    o = align_up(o + 8 * ntile + 256, 256);    // [0]=ticket, [1]=total, from word 32: 64-bit descriptors
        L.fsort_temp = o;    o = align_up(o + sort_temp_bytes_u32(BF), 256);
        L.end = o;
        return L;
    }
};

struct TriFaceLayout {
    FaceBinLayout bin;
    size_t records, total;
    __host__ static TriFaceLayout make(size_t BF)
    {
        TriFaceLayout L;
        L.bin = FaceBinLayout::make(BF);
        size_t o = L.bin.end;
        L.records = o;       o = align_up(o + sizeof(TriRecord) * BF, 256);
        L.total = o + 256;
        return L;
    }
};

// Backward scratch of the tri renderer (dmr_tri_backward's `workspace`), zeroed per call.  Not part of the face
// buffer: that one is saved for backward by autograd and must stay read-only.
struct TriBwdLayout {
    size_t grad_stats, grad_vacc, stats_end, total;
    __host__ static TriBwdLayout make(size_t BF, size_t P)
    {
        TriBwdLayout L;
        size_t o = 0;
        L.grad_stats = o;    o = align_up(o + 96 * BF, 256);   // 24 floats per (view, face)
        L.stats_end = o;
        L.grad_vacc = o;     o = align_up(o + 32 * P, 256);    // float4[2][P]: dL_dverts, dL_dvcolor (16-byte aligned for red.v4)
        L.total = o + 256;
        return L;
    }
};

struct TriImageLayout {
    size_t final_T, prev_T, n_contrib, ranges, total;
    __host__ static TriImageLayout make(size_t B, size_t W, size_t H)
    {
        TriImageLayout L;
        size_t BI = B * W * H;
        size_t tiles = B * ((W + DMR_TILE - 1) / DMR_TILE) * ((H + DMR_TILE - 1) / DMR_TILE);
        size_t o = 0;
        L.final_T = o;   o = align_up(o + 4 * BI, 256);
        L.prev_T = o;    o = align_up(o + 4 * BI, 256);
        L.n_contrib = o; o = align_up(o + 4 * BI, 256);
        L.ranges = o;    o = align_up(o + 8 * tiles, 256);
        L.total = o + 256;
        return L;
    }
};

// binning buffer: A = unsorted (duplicate output), B = sorted, then sort temp.  Keys are 32-bit tile ids
// (tile + tiles_per_view * view): the depth half of the reference's 64-bit key is already sorted when the
// instances are emitted (see bin_faces()).
struct BinningLayout {
    size_t keys_unsorted, vals_unsorted, keys_sorted, vals_sorted, sort_temp, total;
    __host__ static BinningLayout make(size_t R);
};

// ---------------------------------------------------------------------------
// stage launchers (host)
// ---------------------------------------------------------------------------
size_t sort_temp_bytes(size_t n);
int sort_pairs(const uint64_t* keys_in, const uint32_t* vals_in, uint64_t* keys_out, uint32_t* vals_out, size_t n,
               int end_bit, void* temp, cudaStream_t stream);
// 32-bit keys; vals_in == nullptr stands for the identity (0, 1, 2, ...); profile == false: no per-kernel
// profile stages (the caller wraps the whole sort in one)
int sort_pairs_u32(const uint32_t* keys_in, const uint32_t* vals_in, uint32_t* keys_out, uint32_t* vals_out, size_t n,
                   int end_bit, void* temp, bool profile, cudaStream_t stream);

// inclusive scan of in[index ? index[i] : i]
int inclusive_scan_u32(const uint32_t* in, const uint32_t* index, uint32_t* out, size_t n,
                       uint32_t* state /* zeroed, 8*ntile + 256 bytes */, int32_t* total_host /* pinned, may be null */,
                       cudaStream_t stream);

// Two-level binning (replaces InclusiveSum + duplicateWithKeys + the 64-bit SortPairs + identifyTileRanges,
// rasterizer_impl.cu:278-338).  The reference sorts R (tile|depth) keys of 32+bit_length(tiles) bits.  An LSD
// radix sort is a chain of stable passes from the least significant digit up, so the same order results from
//   (1) bin_faces:     stable sort of the B*F FACES by their 32-bit depth key, then the scan over
//                      tiles_touched in that order (R and the instance ranges);
//   (2) bin_instances: emission of the instances in depth order (key = tile id only) and a stable sort on
//                      the bit_length(tiles) tile bits -- 1-3 eight-bit passes over 8-byte pairs instead of
//                      6-7 passes over 12-byte pairs; then the tile ranges.
// Equal (tile, depth) pairs keep ascending b*F+f order in both formulations (stable sorts all the way).
struct SortPre;
// bin_faces_begin zeroes the scan / face-sort control words (one memset) and returns the handle the
// face-preprocess kernel needs to accumulate the depth-key histograms as a by-product (radix_sort.cuh)
int bin_faces_begin(size_t BF, void* face_buffer, const FaceBinLayout& L, SortPre* face_sort, cudaStream_t stream);
// Above this many faces the by-product histogram costs more than it saves (every block of the face kernel
// flushes up to 1024 bins with global atomics: +51 us at 4 M faces against a 20 us histogram kernel); below it
// the two saved launches win (C1/C2: -15 us).
#define DMR_FUSED_FACE_HIST_MAX (1u << 20)
// same for the tile sort's histogram in duplicate_kernel (C4 with 8 views, R = 16.8 M: +209 us fused)
#define DMR_FUSED_TILE_HIST_MAX (1u << 21)
int bin_faces(size_t BF, void* face_buffer, const FaceBinLayout& L, int32_t* num_rendered_host, cudaStream_t stream);
int bin_instances(int B, int F, int W, int H, size_t R, const void* face_buffer, const FaceBinLayout& L,
                  void* binning_buffer, uint2* ranges /* [B*tiles] */, cudaStream_t stream);

uint32_t higher_msb(uint32_t n);

// image.cu: alpha image and background gradient of either renderer from its image state.  t: tri final_T, tet
// final_log_T (both [B,H,W]); active: tet only ([B,H,W] bytes), nullptr for tri.  image_bg_grad writes dL_dbg[3] and
// needs image_bg_grad_bytes(B) bytes of workspace.
int image_alpha(bool tet, int B, int W, int H, const float* t, const uint8_t* active, float* alpha, cudaStream_t stream);
size_t image_bg_grad_bytes(int B);
int image_bg_grad(bool tet, int B, int W, int H, const float* t, const uint8_t* active, const float* dL_dcolor, float* dL_dbg,
                  void* workspace, cudaStream_t stream);

// image.cu: the face statistics' workspace (12 * B * F bytes: the fixed-point weights, then the hit counts) and the
// conversion of its accumulators into face_weights [B*F] fp32 and face_hits [B*F] int32 (one launch; the caller
// opens the profile stage)
size_t face_weights_bytes(int B, int F);
FaceWeightAcc face_weights_acc(void* workspace, int B, int F);
int face_weights_convert(int B, int F, const FaceWeightAcc& acc, float* face_weights, int* face_hits, cudaStream_t stream);

}  // namespace dmr
