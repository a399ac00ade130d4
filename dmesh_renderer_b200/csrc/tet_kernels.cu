// tet_kernels.cu -- tet renderer: adjacency records, first intersection, ray march.
//
//   tet_build_*_kernel          hoist tet_face_outward_normal (cuda_renderer/auxiliary.h:345-394),
//                               get_face_vert / get_face_vert_color (402-456) and the
//                               face_tets neighbour search (forward.cu:761-767) out of the march
//   tet_jitter_kernel           setup_curand_kernel + jitter of generateRaysCUDA (forward.cu:82-88,120-123)
//   tet_first_intersect_kernel  replaces firstIntersectCUDA (forward.cu:298-445)
//   tet_march_fwd_kernel        replaces TET_FORWARD::renderCUDA (forward.cu:485-815)
//   tet_march_bwd_kernel        replaces TET_BACKWARD::renderCUDA (backward.cu:86-487)
//   tet_march_bwd_cam_kernel,   the same plus gradients with respect to the camera matrices (no reference counterpart)
//   tet_camera_finish_kernel
//   tet_march_bwd_*vert*_kernel the same plus gradients with respect to the vertex positions (no reference counterpart)
//
// Forward images must match the reference to 1e-5, which requires IDENTICAL
// branch decisions along every ray (hit tests, normal signs); all such
// expressions keep the reference's operation order.
#include "tet.cuh"
#include "det.cuh"
#include <curand_kernel.h>
#include <type_traits>

namespace dmr {

// ---------------------------------------------------------------------------
// geometry helpers
// ---------------------------------------------------------------------------

// dot / cross with the contraction nvcc applies to cuda_math.h:1524-1527, 1696-1699 written out
// (fma(z,z', fma(x,x', y*y')) and fma(a,b,-(c*d)), the same forms oracle/oracle.cpp pins): every call
// site then yields the SAME bits for the same inputs, whatever the surrounding code.  The backward
// pass depends on that wherever it recomputes (t,u,v) of a face with the hit test below (the last face of a
// ray, and the re-march beyond the trail): it must get what the forward march got -- the depth term
// (pd - accum_recd) of the opacity gradient amplifies a one-ulp change of t by 1e3..1e4.  (The recorded part of
// a ray replays the forward pass's own (t,u,v) from the trail.)
__device__ __forceinline__ float dot3p(float3 a, float3 b)
{
    return __fmaf_rn(a.z, b.z, __fmaf_rn(a.x, b.x, __fmul_rn(a.y, b.y)));
}
__device__ __forceinline__ float3 cross3p(float3 a, float3 b)
{
    return f3(__fmaf_rn(a.y, b.z, -__fmul_rn(a.z, b.y)), __fmaf_rn(a.z, b.x, -__fmul_rn(a.x, b.z)),
              __fmaf_rn(a.x, b.y, -__fmul_rn(a.y, b.x)));
}

// Moeller-Trumbore with inside test: cuda_renderer/auxiliary.h:265-296.
// tuv is left untouched when denom == 0 (as in the reference).
__device__ __forceinline__ bool ray_tri_hit(float3 ro, float3 rd, float3 p0, float3 p1, float3 p2, float3& tuv)
{
    float3 T = ro - p0;
    float3 E1 = p1 - p0;
    float3 E2 = p2 - p0;
    float3 Pv = cross3p(rd, E2);
    float3 Q = cross3p(T, E1);
    float denom = dot3p(Pv, E1);
    if (denom == 0.0f) return false;
    float inv_denom = 1.0f / denom;
    tuv.x = __fmul_rn(dot3p(Q, E2), inv_denom);
    tuv.y = __fmul_rn(dot3p(Pv, T), inv_denom);
    tuv.z = __fmul_rn(dot3p(Q, rd), inv_denom);
    return (tuv.x >= 0.0f && tuv.y >= 0.0f && tuv.z >= 0.0f && tuv.y + tuv.z <= 1.0f);
}

__device__ __forceinline__ float3 ld3(const float* p) { return f3(p[0], p[1], p[2]); }

// cuda_renderer/auxiliary.h:345-394
__device__ __forceinline__ float3 outward_normal(float3 p0, float3 p1, float3 p2, float3 q0, float3 q1, float3 q2,
                                                 float3 q3)
{
    float3 d1 = p1 - p0;
    float3 d2 = p2 - p0;
    float3 n = cross3(d1, d2);
    float n_norm = sqrtf(dot3(n, n));
    n_norm = fmaxf(n_norm, 0.0001f);
    n = n / n_norm;
    float3 centre = (q0 + q1 + q2 + q3) * 0.25f;
    float3 d = centre - p0;
    float dp = dot3(n, d);
    if (dp > 0.0f) n = -n;
    return n;
}

// ---------------------------------------------------------------------------
// record builders (view independent, once per forward call)
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(128) tet_build_tetrec_kernel(
    int T, const float* __restrict__ verts, const int* __restrict__ faces, const int* __restrict__ tets,
    const int* __restrict__ face_tets, const int* __restrict__ tet_faces, TetRec* __restrict__ out)
{
    griddep_wait();   // programmatic dependent launch: see dmr_launch (common.cuh)
    __shared__ uint4 s_rec[128 * 8];   // 128 B per tet; written per thread, read back coalesced
    const int t0 = blockIdx.x * 128;
    const int t = t0 + threadIdx.x;
    if (t < T) {
        const int4 tv4 = reinterpret_cast<const int4*>(tets)[t];
        const int4 tf = reinterpret_cast<const int4*>(tet_faces)[t];
        const int tv[4] = { tv4.x, tv4.y, tv4.z, tv4.w };
        float3 q[4];
#pragma unroll
        for (int i = 0; i < 4; i++) q[i] = ld3(verts + 3 * (size_t)tv[i]);
        const int fid[4] = { tf.x, tf.y, tf.z, tf.w };
        uint32_t nxt[4];
        float3 nrm[4];
        int loc[4][3];      // tet-local index (0..3) of the side's p0, p1, p2; -1 = not a vertex of this tet
        int opp[4];         // tet-local index of the vertex opposite side k
        bool regular = true;
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const int f = fid[k];
            const int fv[3] = { faces[3 * (size_t)f], faces[3 * (size_t)f + 1], faces[3 * (size_t)f + 2] };
            float3 pp[3];
#pragma unroll
            for (int j = 0; j < 3; j++) pp[j] = ld3(verts + 3 * (size_t)fv[j]);
            nrm[k] = outward_normal(pp[0], pp[1], pp[2], q[0], q[1], q[2], q[3]);
            // forward.cu:761-767
            int nt = -1;
            for (int i = 0; i < 2; i++) {
                int cand = face_tets[2 * (size_t)f + i];
                if (cand == t || cand == -1) continue;
                nt = cand;
                break;
            }
            nxt[k] = (uint32_t)(nt + 1);
            // which tet vertex is p_j?  by id, else by bitwise-equal position (duplicated vertices)
#pragma unroll
            for (int j = 0; j < 3; j++) {
                int l = -1;
#pragma unroll
                for (int i = 3; i >= 0; i--)
                    if (fv[j] == tv[i] || (pp[j].x == q[i].x && pp[j].y == q[i].y && pp[j].z == q[i].z)) l = i;
                loc[k][j] = l;
            }
            const int l0 = loc[k][0], l1 = loc[k][1], l2 = loc[k][2];
            if (l0 < 0 || l1 < 0 || l2 < 0 || l0 == l1 || l0 == l2 || l1 == l2) { regular = false; opp[k] = 0; }
            else opp[k] = 6 - l0 - l1 - l2;
        }
        // the four sides must be opposite four different vertices
        if (regular && ((1 << opp[0]) | (1 << opp[1]) | (1 << opp[2]) | (1 << opp[3])) != 0xF) regular = false;
        float3 vout[4];
#pragma unroll
        for (int k = 0; k < 4; k++) {
            uint32_t code = 0xFu;
            vout[k] = q[k];
            if (regular) {
                vout[k] = q[0];
#pragma unroll
                for (int i = 1; i < 4; i++) if (opp[k] == i) vout[k] = q[i];
                // position of p0 / p1 inside cyc = (vert[(k+1)&3], vert[(k+2)&3], vert[(k+3)&3])
                int a = 0, bb = 0;
#pragma unroll
                for (int j = 1; j <= 3; j++) {
                    if (opp[(k + j) & 3] == loc[k][0]) a = j - 1;
                    if (opp[(k + j) & 3] == loc[k][1]) bb = j - 1;
                }
                code = (uint32_t)(a | (bb << 2));
            }
            nxt[k] |= code << 28;
        }
        uint4* o = s_rec + threadIdx.x * 8;
        o[0] = make_uint4(fid[0], fid[1], fid[2], fid[3]);
        o[1] = make_uint4(nxt[0], nxt[1], nxt[2], nxt[3]);
        o[2] = make_uint4(__float_as_uint(vout[0].x), __float_as_uint(vout[0].y), __float_as_uint(vout[0].z), __float_as_uint(vout[1].x));
        o[3] = make_uint4(__float_as_uint(vout[1].y), __float_as_uint(vout[1].z), __float_as_uint(vout[2].x), __float_as_uint(vout[2].y));
        o[4] = make_uint4(__float_as_uint(vout[2].z), __float_as_uint(vout[3].x), __float_as_uint(vout[3].y), __float_as_uint(vout[3].z));
        o[5] = make_uint4(__float_as_uint(nrm[0].x), __float_as_uint(nrm[0].y), __float_as_uint(nrm[0].z), __float_as_uint(nrm[1].x));
        o[6] = make_uint4(__float_as_uint(nrm[1].y), __float_as_uint(nrm[1].z), __float_as_uint(nrm[2].x), __float_as_uint(nrm[2].y));
        o[7] = make_uint4(__float_as_uint(nrm[2].z), __float_as_uint(nrm[3].x), __float_as_uint(nrm[3].y), __float_as_uint(nrm[3].z));
    }
    __syncthreads();
    const int nvalid = min(128, T - t0);
    uint4* dst = reinterpret_cast<uint4*>(out + t0);
    for (int i = threadIdx.x; i < nvalid * 8; i += 128) dst[i] = s_rec[i];
}

__global__ void __launch_bounds__(256) tet_build_shade_kernel(
    int F, const int* __restrict__ faces, const float* __restrict__ verts_color, const float* __restrict__ faces_opacity,
    const int* __restrict__ face_tets, TetShade* __restrict__ out)
{
    griddep_wait();   // programmatic dependent launch: see dmr_launch (common.cuh)
    int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= F) return;
    const int a = faces[3 * (size_t)f], b = faces[3 * (size_t)f + 1], c = faces[3 * (size_t)f + 2];
    float3 c0 = ld3(verts_color + 3 * (size_t)a), c1 = ld3(verts_color + 3 * (size_t)b), c2 = ld3(verts_color + 3 * (size_t)c);
    uint4* o = reinterpret_cast<uint4*>(out + f);
    o[0] = make_uint4(__float_as_uint(c0.x), __float_as_uint(c0.y), __float_as_uint(c0.z), __float_as_uint(c1.x));
    o[1] = make_uint4(__float_as_uint(c1.y), __float_as_uint(c1.z), __float_as_uint(c2.x), __float_as_uint(c2.y));
    o[2] = make_uint4(__float_as_uint(c2.z), __float_as_uint(faces_opacity[f]), __float_as_uint(logf(1.0f - faces_opacity[f])), a);
    // log(1 - opacity) is a per-face constant of the march (forward.cu:636-642, backward.cu:272-279):
    // same logf on the same input, evaluated once per face instead of once per step
    o[3] = make_uint4(b, c, face_tets[2 * (size_t)f], face_tets[2 * (size_t)f + 1]);
}

int tet_build_records(int P, int F, int T, const float* verts, const int* faces, const float* verts_color,
                      const float* faces_opacity, const int* tets, const int* face_tets, const int* tet_faces,
                      TetRec* tet_rec, TetShade* shade, cudaStream_t stream)
{
    (void)P;
    ProfScope prof(ST_TET_RECORDS, stream);
    if (T > 0 && F > 0 && tet_rec && shade) count_launch(1);   // two kernels under one scope
    if (T > 0 && tet_rec) {
        DMR_CUDA(dmr_launch(tet_build_tetrec_kernel, dim3((T + 127) / 128), dim3(128), 0, stream, T, verts, faces, tets, face_tets, tet_faces, tet_rec));
        DMR_LAUNCH_CHECK("tet_build_tetrec_kernel");
    }
    if (F > 0 && shade) {
        DMR_CUDA(dmr_launch(tet_build_shade_kernel, dim3((F + 255) / 256), dim3(256), 0, stream, F, faces, verts_color, faces_opacity, face_tets, shade));
        DMR_LAUNCH_CHECK("tet_build_shade_kernel");
    }
    return 0;
}

// ---------------------------------------------------------------------------
// jittered pixel coordinates (ray_random_seed > 0): XORWOW, sequence = pixel index
// forward.cu:82-88, 120-123.  Stored (8 B/px) so that first-intersect, march and
// backward see the same ray without re-running curand_init three times.
// The sequence counts pixels from view `first_view` of the whole job, (first_view + b)*H*W + y*W + x, so a view
// gets the same rays whichever call (or rank) renders it; first_view = 0 is the reference's pixel index.
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256) tet_jitter_kernel(int BI, int W, int H, int seed, int first_view,
                                                         float2* __restrict__ jitter)
{
    griddep_wait();   // programmatic dependent launch: see dmr_launch (common.cuh)
    int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= BI) return;
    curandState st;
    curand_init(seed, (unsigned long long)first_view * W * H + (unsigned long long)idx, 0, &st);
    int pixel_id = idx % (W * H);
    int pixel_x = pixel_id % W, pixel_y = pixel_id / W;
    float2 o;
    o.x = pixel_x - 0.5f + (0.5f * curand_uniform(&st));
    o.y = pixel_y - 0.5f + (0.5f * curand_uniform(&st));
    jitter[idx] = o;
}

int tet_jitter(int B, int W, int H, int seed, int first_view, float2* jitter, cudaStream_t stream)
{
    int BI = B * W * H;
    if (BI <= 0) return 0;
    ProfScope prof(ST_TET_JITTER, stream);
    DMR_CUDA(dmr_launch(tet_jitter_kernel, dim3((BI + 255) / 256), dim3(256), 0, stream, BI, W, H, seed, first_view,
                        jitter));
    DMR_LAUNCH_CHECK("tet_jitter_kernel");
    return 0;
}

__device__ __forceinline__ void tet_pixel_ray(const TetParams& p, int b, uint32_t px, uint32_t py, size_t bpix,
                                              float3& ro, float3& rd)
{
    float fx = px + 0.5f, fy = py + 0.5f;
    if (p.jitter) { float2 j = p.jitter[bpix]; fx = j.x; fy = j.y; }
    pixel_ray<true>(p.inv_mv + 16 * b, p.inv_proj + 16 * b, fx, fy, p.W, p.H, ro, rd);
}

// ---------------------------------------------------------------------------
// first intersection: per tile, faces sorted by min depth
// ---------------------------------------------------------------------------
#define FI_THREADS 256
__device__ __forceinline__ void tet_first_finish(const TetParams& p, int b, size_t bpix, int first_face, float3 rd);

// Face-parallel search.  One CTA per 16x16 tile; per round 256 instances of the tile list are staged
// (one per thread) and EVERY THREAD TAKES ONE FACE: it walks the pixels of the face's screen bounding
// box inside the tile that are still searching, runs the reference's ray/triangle test and merges hits
// into the pixel's slot with a 64-bit shared-memory atomicMin on (t bits << 32 | list position) --
// the lexicographic minimum is exactly what the reference's sequential "cur < min_T" scan keeps (first
// face in list order among equal t).  Then every thread folds the round's winner of ITS pixel into its
// running best and applies the reference's early-out (forward.cu:388-391) at round granularity.
//
// Why: the reference (and the first two versions of this kernel) walk the list once per pixel block
// with one warp -- a serial chain whose length is the whole tile list (5-20 k faces at C3) for every
// block that contains a pixel the mesh does not cover.  The kernel's duration was the latency of that
// chain in a few hundred silhouette tiles (688 us at C3 with 14% achieved occupancy and 45 M warp
// instructions, i.e. 40 us of issue work).  Taking faces instead of pixels as the parallel axis makes a
// round 256 independent tests wide.
//
// Equivalence with the sequential scan: faces are sorted by min depth, a face is skipped by the reference
// only when its min depth exceeds the max depth of the current best hit, and NDC depth is monotone in t
// along a ray, so the skipped faces cannot hold the minimum; the result is the argmin of t over all hit
// faces (ties: list order) either way.  The early-out is applied between rounds, and a round winner that
// the reference would not have reached any more (min depth beyond the previous best's max depth) is
// discarded like the reference does.
__global__ void __launch_bounds__(FI_THREADS) tet_first_intersect_kernel(TetParams p)
{
    griddep_wait();   // programmatic dependent launch: see dmr_launch (common.cuh)
    __shared__ uint4 s_rec[FI_THREADS * 3];          // p0 p1 p2 | min_depth max_depth bbox_x
    __shared__ uint32_t s_bby[FI_THREADS];
    __shared__ int s_face[FI_THREADS];
    __shared__ unsigned long long s_best[FI_THREADS];
    __shared__ float4 s_rd[FI_THREADS];
    __shared__ uint32_t s_open[DMR_TILE];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    // fi_split CTAs share a tile: CTA `part` takes rounds part, part + fi_split, ... of the tile list and the
    // partial results meet in a global 64-bit atomicMin per pixel (tet_first_resolve_kernel turns the winner
    // into first_face / first_tet).  The kernel's duration is the longest tile list (a few hundred silhouette
    // tiles at C3); splitting it shortens exactly that chain.  `part` is the SLOWEST grid dimension: the
    // part-0 CTAs of all tiles are scheduled first, so that by the time a later part starts, the interior
    // tiles (finished by part 0 in one or two rounds) have published their closing depths and it stops at once.
    const int split = p.fi_split, part = (int)(blockIdx.z / (unsigned)p.B), b = (int)(blockIdx.z % (unsigned)p.B);
    const int tile_x = blockIdx.x;
    const int tiles_x = gridDim.x, tiles_y = gridDim.y;
    const uint32_t tx0 = tile_x * DMR_TILE, ty0 = blockIdx.y * DMR_TILE;
    const uint32_t px = tx0 + (tid & 15);
    const uint32_t py = ty0 + (tid >> 4);
    const bool inside = px < (uint32_t)p.W && py < (uint32_t)p.H;
    const size_t bpix = (size_t)b * p.W * p.H + (size_t)py * p.W + px;

    float3 ro = f3(p.inv_mv[16 * b + 12], p.inv_mv[16 * b + 13], p.inv_mv[16 * b + 14]);   // same for every pixel
    float3 rd = f3(0, 0, 1);
    if (inside) tet_pixel_ray(p, b, px, py, bpix, ro, rd);
    s_rd[tid] = make_float4(rd.x, rd.y, rd.z, 0.0f);
    ro = f3(p.inv_mv[16 * b + 12], p.inv_mv[16 * b + 13], p.inv_mv[16 * b + 14]);

    const uint2 range = p.ranges[(size_t)b * tiles_x * tiles_y + blockIdx.y * tiles_x + tile_x];
    const int total = (int)(range.y - range.x);
    const int rounds = (total + FI_THREADS - 1) / FI_THREADS;

    float min_T = -1.0f, min_T_max_depth = -1.0f;
    int first_face = -1;
    uint32_t first_pos = 0;     // list position of the best hit (split mode)
    bool closed = !inside;

    // register-staged prefetch of the next round
    uint4 n0 = make_uint4(0, 0, 0, 0), n1 = n0, n2 = n0;
    uint32_t nby = 0;
    int nface = 0;
    auto fetch = [&](int r) {
        const uint32_t pos = range.x + (uint32_t)r * FI_THREADS + tid;
        if (r < rounds && pos < range.y) {
            nface = (int)p.face_list[pos];
            const uint4* src = reinterpret_cast<const uint4*>(p.face_rec + (size_t)b * p.F + nface);
            n0 = src[0]; n1 = src[1]; n2 = src[2];
            nby = src[3].x;
        }
    };
    fetch(part);

    for (int r = part; r < rounds; r += split) {
        s_rec[tid * 3 + 0] = n0; s_rec[tid * 3 + 1] = n1; s_rec[tid * 3 + 2] = n2;
        s_bby[tid] = nby;
        s_face[tid] = nface;
        s_best[tid] = ~0ull;
        __syncthreads();
        // forward.cu:388-391 at round granularity: nothing from this round on can beat the best hit
        if (!closed && min_T >= 0.0f && __uint_as_float(s_rec[2].y) > min_T_max_depth) closed = true;
        // split mode: ... nor a hit found by one of the other CTAs of this tile (smallest max depth of any hit
        // so far; a face whose min depth lies beyond it cannot hold the first intersection)
        if (!closed && split > 1 && __uint_as_float(s_rec[2].y) > __uint_as_float(__ldcg(p.fi_close + bpix))) closed = true;
        {
            const unsigned open = __ballot_sync(0xffffffffu, !closed);   // a warp holds tile rows 2*warp, 2*warp+1
            if (lane == 0) { s_open[2 * warp] = open & 0xffffu; s_open[2 * warp + 1] = open >> 16; }
        }
        if (__syncthreads_count(!closed) == 0) break;
        fetch(r + split);

        const int cnt = min(FI_THREADS, total - r * FI_THREADS);
        // (fetch(r+1) overwrote the staging registers; this round's face is read back from shared memory)
        if (tid < cnt) {
            const uint4 q0 = s_rec[tid * 3 + 0], q1 = s_rec[tid * 3 + 1], q2 = s_rec[tid * 3 + 2];
            const uint32_t bbx = q2.w, bby = s_bby[tid];
            const int x0 = max((int)(bbx & 0xffffu), (int)tx0), x1 = min((int)(bbx >> 16), (int)tx0 + DMR_TILE - 1);
            const int y0 = max((int)(bby & 0xffffu), (int)ty0), y1 = min((int)(bby >> 16), (int)ty0 + DMR_TILE - 1);
            if (x0 <= x1) {
                const float3 p0 = f3(__uint_as_float(q0.x), __uint_as_float(q0.y), __uint_as_float(q0.z));
                const float3 p1 = f3(__uint_as_float(q0.w), __uint_as_float(q1.x), __uint_as_float(q1.y));
                const float3 p2 = f3(__uint_as_float(q1.z), __uint_as_float(q1.w), __uint_as_float(q2.x));
                const uint32_t xmask = ((2u << (x1 - (int)tx0)) - 1u) & ~((1u << (x0 - (int)tx0)) - 1u);
                for (int y = y0; y <= y1; y++) {
                    uint32_t m = s_open[y - (int)ty0] & xmask;
                    while (m) {
                        const int xi = __ffs(m) - 1;
                        m &= m - 1;
                        const int pix = (y - (int)ty0) * DMR_TILE + xi;
                        const float4 d4 = s_rd[pix];
                        float3 tuv;
                        if (!ray_tri_hit(ro, f3(d4.x, d4.y, d4.z), p0, p1, p2, tuv)) continue;
                        const uint32_t tb = tuv.x == 0.0f ? 0u : __float_as_uint(tuv.x);   // t >= 0: bits are monotone
                        atomicMin(&s_best[pix], ((unsigned long long)tb << 32) | (unsigned)tid);
                    }
                }
            }
        }
        __syncthreads();
        if (!closed) {
            const unsigned long long key = s_best[tid];
            if (key != ~0ull) {
                const int pos = (int)(key & 0xffffffffu);
                const float cur = __uint_as_float((uint32_t)(key >> 32));
                const uint4 q2 = s_rec[pos * 3 + 2];
                // the reference stops in front of a face whose min depth exceeds the best hit's max depth
                if (min_T >= 0.0f && __uint_as_float(q2.y) > min_T_max_depth) closed = true;
                else if (min_T < 0.0f || cur < min_T) {
                    min_T = cur;
                    min_T_max_depth = __uint_as_float(q2.z);
                    first_face = s_face[pos];
                    first_pos = (uint32_t)(r * FI_THREADS + pos);
                    if (split > 1) atomicMin(p.fi_close + bpix, q2.z);   // max depth bits (non-negative float)
                }
            }
        }
        __syncthreads();
    }

    if (!inside) return;
    if (split > 1) {   // partial result: (t, list position) into the pixel's global slot
        if (first_face >= 0) {
            const uint32_t tb = min_T == 0.0f ? 0u : __float_as_uint(min_T);
            atomicMin(p.fi_key + bpix, ((unsigned long long)tb << 32) | first_pos);
        }
        return;
    }
    tet_first_finish(p, b, bpix, first_face, rd);
}

// first_tet of a pixel (forward.cu:419-444: the adjacent tet whose outward normal opposes the ray) + stores
__device__ __forceinline__ void tet_first_finish(const TetParams& p, int b, size_t bpix, int first_face, float3 rd)
{
    (void)b;
    int first_tet = -1;
    if (first_face >= 0) {
        const TetShade* sh = p.shade + first_face;
        const int cand[2] = { sh->t0, sh->t1 };
        for (int i = 0; i < 2; i++) {
            int tet_id = cand[i];
            if (tet_id < 0) continue;
            const TetRec* tr = p.tet_rec + tet_id;
            float3 n = f3(0, 0, 0);
            bool found = false;
#pragma unroll
            for (int k = 0; k < 4; k++)
                if (!found && tr->face[k] == first_face) { n = f3(tr->nrm[k][0], tr->nrm[k][1], tr->nrm[k][2]); found = true; }
            if (!found) continue;   // inconsistent adjacency tables
            if (dot3p(n, rd) < 0.0f) first_tet = tet_id;
        }
    }
    p.first_face[bpix] = first_face;
    p.first_tet[bpix] = first_tet;
}

// split mode: winner of the pixel's partial results -> first_face, first_tet
__global__ void __launch_bounds__(256) tet_first_resolve_kernel(TetParams p)
{
    griddep_wait();   // programmatic dependent launch: see dmr_launch (common.cuh)
    const int b = blockIdx.z;
    const uint32_t px = blockIdx.x * 16 + (threadIdx.x & 15), py = blockIdx.y * 16 + (threadIdx.x >> 4);
    if (!(px < (uint32_t)p.W && py < (uint32_t)p.H)) return;
    const size_t bpix = (size_t)b * p.W * p.H + (size_t)py * p.W + px;
    const unsigned long long key = p.fi_key[bpix];
    int first_face = -1;
    if (key != ~0ull) {
        const uint2 range = p.ranges[((size_t)b * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x];
        first_face = (int)p.face_list[range.x + (uint32_t)(key & 0xffffffffu)];
    }
    float3 ro, rd;
    tet_pixel_ray(p, b, px, py, bpix, ro, rd);
    tet_first_finish(p, b, bpix, first_face, rd);
}

int tet_first_intersect(const TetParams& p, cudaStream_t stream)
{
    const int tx = (p.W + DMR_TILE - 1) / DMR_TILE, ty = (p.H + DMR_TILE - 1) / DMR_TILE;
    ProfScope prof(ST_TET_FIRST, stream);
    if (p.fi_split > 1) {
        count_launch(1);   // two kernels under one scope
        DMR_CUDA(cudaMemsetAsync(p.fi_key, 0xff, 12 * (size_t)p.B * p.W * p.H, stream));   // fi_key + fi_close
    }
    DMR_CUDA(dmr_launch(tet_first_intersect_kernel, dim3(tx, ty, p.B * p.fi_split), dim3(FI_THREADS), 0, stream, p));
    DMR_LAUNCH_CHECK("tet_first_intersect_kernel");
    if (p.fi_split > 1) {
        DMR_CUDA(dmr_launch(tet_first_resolve_kernel, dim3(tx, ty, p.B), dim3(256), 0, stream, p));
        DMR_LAUNCH_CHECK("tet_first_resolve_kernel");
    }
    return 0;
}

// ---------------------------------------------------------------------------
// forward march
// ---------------------------------------------------------------------------
// The march is independent per pixel (no shared memory, no tile lists) and its cost per ray has a
// long tail (rays along the cube diagonal cross several times more faces than the mean), so it is
// launched as many small CTAs: 64 threads = 8x8 pixels = two 8x4 warps.
constexpr int MARCH_THREADS = 64;
constexpr int MARCH_ROWS = MARCH_THREADS / 8;   // pixel rows of a CTA: 8 columns x 4 rows per warp
// 10 CTAs/SM = 96 registers (forward march at C3 after the depth computation left the loop: 8 CTAs / 112 registers
// 820 us, 10 / 96 (2 spill slots) 772 us, 12 / 80 (14 spill accesses per step) 783 us; round 1: 64 registers 947 us)
constexpr int MARCH_MIN_BLOCKS = 10;

struct TetStep {   // result of looking for the exit (or entry) face of a tet
    int face, tet;
    float rt, iu, iv;
    bool ok;
    bool opposite;   // some other side is hit with the OPPOSITE normal sign (see the face trail)
    bool irregular;  // IRR = false only: a side of an irregular tet was met (ok is false; the caller re-marches the ray)
};

// Among the sides of `tet` other than `curr_face`, the unique one hit by the ray whose
// outward normal has the requested sign against the ray: forward.cu:672-768 (EXIT: normal
// along the ray) and backward.cu:382-477 (ENTRY: normal against the ray).
// (Measured and rejected: prefetching the records of all candidate next tets / faces into L2 as soon
// as the current tet's ids are known made the march SLOWER -- fwd 0.91 -> 1.03 ms, bwd 1.51 -> 2.25 ms
// at C3: the extra address arithmetic and L2 requests cost more than the latency they hide.)
// one of three values by a 2-bit index (0, 1, 2): two selects
__device__ __forceinline__ float sel3(int i, float a, float b, float c) { return i == 2 ? c : (i == 1 ? b : a); }
__device__ __forceinline__ float3 sel3(int i, float3 a, float3 b, float3 c)
{
    return f3(sel3(i, a.x, b.x, c.x), sel3(i, a.y, b.y, c.y), sel3(i, a.z, b.z, c.z));
}

// NDC depth of the point ro + t * rd (forward.cu:629-632, backward.cu:262-266: the point is carried through the
// model-view and the projection matrix and z / clamp(w) is kept).  Both clip coordinates are affine in t with
// per-pixel coefficients -- z_clip = az + t * bz, w_clip = aw + t * bw, from the z and w rows of proj * mv -- so a
// march step costs two fused multiply-adds and a reciprocal instead of re-reading both matrices: the 28 uniform
// loads per step were 18 % of the forward march's L1 wavefronts and the L1 data pipe is its busiest unit (67 % of
// peak at C3).  Same real number as the reference's chain, rounded differently (~1e-7 relative; the depth image
// is compared at 1e-5).
struct TetDepth { float az, bz, aw, bw; };
// z and w rows of proj * mv over the first three rows of mv (the bottom row of mv never enters: xform43)
__device__ __forceinline__ void tet_depth_rows(const float* __restrict__ mv, const float* __restrict__ pj, float rz[4], float rw[4])
{
#pragma unroll
    for (int k = 0; k < 4; k++) {
        rz[k] = pj[2] * mv[4 * k] + pj[6] * mv[4 * k + 1] + pj[10] * mv[4 * k + 2];
        rw[k] = pj[3] * mv[4 * k] + pj[7] * mv[4 * k + 1] + pj[11] * mv[4 * k + 2];
    }
    rz[3] += pj[14]; rw[3] += pj[15];
}
__device__ __forceinline__ TetDepth tet_depth_setup(const float* __restrict__ mv, const float* __restrict__ pj, float3 ro, float3 rd)
{
    float rz[4], rw[4];
    tet_depth_rows(mv, pj, rz, rw);
    TetDepth d;
    d.az = rz[0] * ro.x + rz[1] * ro.y + rz[2] * ro.z + rz[3];
    d.bz = rz[0] * rd.x + rz[1] * rd.y + rz[2] * rd.z;
    d.aw = rw[0] * ro.x + rw[1] * ro.y + rw[2] * ro.z + rw[3];
    d.bw = rw[0] * rd.x + rw[1] * rd.y + rw[2] * rd.z;
    return d;
}
__device__ __forceinline__ float tet_depth_at(const TetDepth& d, float t)
{
    const float pw = 1.0f / clamp_w(d.aw + t * d.bw);
    return (d.az + t * d.bz) * pw;
}
// The ~1e-7 above is relative to the clip coordinates' magnitude at the camera, not to w: both chains cancel the
// camera's own offset (w = 0 at the eye), each leaving a different rounding error of about eps * |rw . ro| in w and
// likewise in z, so they part by roughly eps * (m_z + |depth| m_w) / |w|.  Hit points close to the camera plane --
// a camera inside the mesh -- make that visible in the depth image (measured 1.1e-5 on a Delaunay mesh seen from
// inside, tests/test_gpu_tet_general_meshes.py).  The forward march takes the reference's chain for such steps:
// tet_depth_scale gives max(m_z, m_w) of a view (uniform: ro is the eye), and a step whose |w| is below
// (1 + |depth|) * scale / 16 -- where the two chains may part by more than ~16 * 4 eps ~ 4e-6 -- is evaluated again
// by tet_depth_exact.  Cameras outside the mesh never need it (C3: |w| >= 2.2 against at most 2 * 8 / 16 = 1).
__device__ __forceinline__ float tet_depth_scale(const float* __restrict__ mv, const float* __restrict__ pj,
                                                 const float* __restrict__ inv_mv)
{
    float rz[4], rw[4];
    tet_depth_rows(mv, pj, rz, rw);
    float mz = fabsf(rz[3]), mw = fabsf(rw[3]);
#pragma unroll
    for (int k = 0; k < 3; k++) { mz += fabsf(rz[k] * inv_mv[12 + k]); mw += fabsf(rw[k] * inv_mv[12 + k]); }
    return fmaxf(mz, mw) * (1.0f / 16.0f);
}
// forward.cu:628-631 as the reference evaluates it (second pass of the forward march only: the first pass hands such
// rays over, as it does rays through irregular tets -- a call in its loop costs it spills, the march is register-bound)
__device__ __forceinline__ float tet_depth_exact(const float* __restrict__ mv, const float* __restrict__ pj, float3 ro,
                                              float3 rd, float t)
{
    const float3 pt = ro + (rd * t);
    const float4 pn = xform44(xform43(pt, mv), pj);
    const float pw = 1.0f / clamp_w(pn.w);
    return pn.z * pw;
}

// Hit test of one side of an IRREGULAR tet (TetRec code 0xF: the side is not made of the tet's own four vertices --
// inconsistent input tables, or two vertices of the tet coincide -- so the compact record cannot present its
// vertices).  The reference gathers the side's vertices through faces[] / verts[] whatever the tet looks like
// (forward.cu:700-722); the per-(view, face) record holds exactly that triangle, in faces[] order.  Rare and
// deliberately out of line -- and even so the call costs the forward march 10 % (844 against 768 us at C3: the
// kernel is register-bound), so the forward march runs in two passes: tet_step<EXIT, false> only REPORTS an
// irregular side, the ray is given up and marked, and a second launch of the kernel, instantiated with the slow
// path, re-marches the marked rays from their first face (no rays: the launch costs ~3 us).
__device__ __noinline__ bool tet_side_hit_irregular(const TetFaceRec* __restrict__ face_rec, float3 ro, float3 rd, float3* tuv)
{
    const float* w = reinterpret_cast<const float*>(face_rec);
    float3 r = f3(0, 0, 0);
    const bool hit = ray_tri_hit(ro, rd, f3(w[0], w[1], w[2]), f3(w[3], w[4], w[5]), f3(w[6], w[7], w[8]), r);
    *tuv = r;
    return hit;
}

template <bool EXIT, bool IRR>
__device__ __forceinline__ TetStep tet_step(const TetParams& p, int b, const TetRec* __restrict__ tr, int curr_face,
                                            float3 ro, float3 rd)
{
    TetStep s;
    s.ok = true;
    s.irregular = false;
    s.face = -1; s.tet = -1; s.rt = 0; s.iu = 0; s.iv = 0;
    const uint4* r4 = reinterpret_cast<const uint4*>(tr);
    const uint4 fid = r4[0], nxt = r4[1];
    const float4 a0 = reinterpret_cast<const float4*>(tr)[2], a1 = reinterpret_cast<const float4*>(tr)[3];
    const float4 a2 = reinterpret_cast<const float4*>(tr)[4], n0 = reinterpret_cast<const float4*>(tr)[5];
    const float4 n1 = reinterpret_cast<const float4*>(tr)[6], n2 = reinterpret_cast<const float4*>(tr)[7];
    const int f[4] = { (int)fid.x, (int)fid.y, (int)fid.z, (int)fid.w };
    const uint32_t nx[4] = { nxt.x, nxt.y, nxt.z, nxt.w };
    const float3 v[4] = { f3(a0.x, a0.y, a0.z), f3(a0.w, a1.x, a1.y), f3(a1.z, a1.w, a2.x), f3(a2.y, a2.z, a2.w) };
    const float3 nr[4] = { f3(n0.x, n0.y, n0.z), f3(n0.w, n1.x, n1.y), f3(n1.z, n1.w, n2.x), f3(n2.y, n2.z, n2.w) };
    int cnt = 0, hits = 0;
    bool have_curr = false;
    s.opposite = false;
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const float dn = dot3p(nr[k], rd);
        if (f[k] == curr_face) {
            // the face we stand on must face the other way (error case 2)
            if (!have_curr) { if (EXIT ? (dn >= 0.0f) : (dn <= 0.0f)) s.ok = false; }
            have_curr = true;
            continue;
        }
        cnt++;
        const int code = (int)(nx[k] >> 28);
        float3 tuv;
        bool hit;
        if (code == 0xF) {   // irregular tet (see TetRec): the side's own vertices, as the reference gathers them
            if (!IRR) { s.ok = false; s.irregular = true; continue; }
            hit = tet_side_hit_irregular(p.face_rec + (size_t)b * p.F + f[k], ro, rd, &tuv);
        } else {
            const int ia = code & 3, ib = code >> 2, ic = 3 - ia - ib;
            const float3 A = v[(k + 1) & 3], B = v[(k + 2) & 3], C = v[(k + 3) & 3];
            hit = ray_tri_hit(ro, rd, sel3(ia, A, B, C), sel3(ib, A, B, C), sel3(ic, A, B, C), tuv);
        }
        if (hit && (EXIT ? (dn > 0.0f) : (dn < 0.0f))) {
            s.face = f[k]; s.tet = (int)(nx[k] & 0x0fffffffu) - 1;
            s.rt = tuv.x; s.iu = tuv.y; s.iv = tuv.z;
            hits++;
        }
        if (hit && (EXIT ? (dn < 0.0f) : (dn > 0.0f))) s.opposite = true;
    }
    if (cnt != 3) s.ok = false;      // error case 1
    if (hits != 1) s.ok = false;     // error case 3
    return s;
}

// Loop shape: at the top of a step both the face to composite (curr_face) and the tet to leave
// (curr_tet) are known, so the shading record and the adjacency record are loaded TOGETHER (one memory
// latency per step; the reference, and the first version of this kernel, composite first and only then
// start the dependent gathers of the tet), and the exit search runs unconditionally next to the
// compositing arithmetic -- two independent dependency chains in one basic block.  Its result is
// simply discarded when the ray terminates in this step; the decisions are taken in the reference's
// order (forward.cu:645-648, 667-670, 687-759).
// (Measured and rejected at the end of round 2: warp-cooperative staging of the adjacency records.  ncu shows no sharing
// between the lanes of a warp -- 128 sectors per warp and step: every lane is in its own tet -- so the eight LDG.128 of
// a lane cost one L1 wavefront per lane each, ~190 of the ~200 wavefronts of a step.  Copying the warp's 32 records to
// shared memory with eight cp.async rounds in which eight consecutive lanes fetch ONE record's line, then eight
// conflict-free LDS.128 per lane (144-byte stride), halves the wavefronts -- and makes the march 4.5 % SLOWER, C3
// 780 -> 815 us: the loop becomes warp-uniform with a copy / wait / read-back round trip in every step's dependent
// chain, and the L1 data pipe at 56 % was not what the step waits for.)
#define DMR_TET_REDO 2   // value of active[] between the two passes of the forward march: ray met an irregular tet
template <bool IRR>      // IRR = true: second pass, only the rays the first pass marked (see tet_side_hit_irregular)
__global__ void __launch_bounds__(MARCH_THREADS, MARCH_MIN_BLOCKS) tet_march_fwd_kernel(TetParams p)
{
    griddep_wait();   // programmatic dependent launch: see dmr_launch (common.cuh)
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int b = blockIdx.z;
    const uint32_t px = blockIdx.x * 8 + (lane & 7);
    const uint32_t py = blockIdx.y * MARCH_ROWS + warp * 4 + (lane >> 3);
    if (!(px < (uint32_t)p.W && py < (uint32_t)p.H)) return;
    const size_t HW = (size_t)p.W * p.H;
    const size_t BI = (size_t)p.B * HW;
    const size_t pix = (size_t)py * p.W + px;
    const size_t bpix = (size_t)b * HW + pix;
    if (IRR && p.active[bpix] != DMR_TET_REDO) return;
    bool redo = false;

    float3 ro, rd;
    tet_pixel_ray(p, b, px, py, bpix, ro, rd);
    const TetDepth dep = tet_depth_setup(p.mv + 16 * b, p.proj + 16 * b, ro, rd);
    const float dep_scale = tet_depth_scale(p.mv + 16 * b, p.proj + 16 * b, p.inv_mv + 16 * b);

    const int first_face = p.first_face[bpix], first_tet = p.first_tet[bpix];
    bool done = false;
    float rt = 0.0f, iu = 0.0f, iv = 0.0f;
    if (first_face == -1 || first_tet == -1) done = true;
    else {
        const float* w = reinterpret_cast<const float*>(p.face_rec + (size_t)b * p.F + first_face);
        float3 tuv = f3(0, 0, 0);
        ray_tri_hit(ro, rd, f3(w[0], w[1], w[2]), f3(w[3], w[4], w[5]), f3(w[6], w[7], w[8]), tuv);
        rt = tuv.x; iu = tuv.y; iv = tuv.z;
    }

    float3 C = f3(0, 0, 0);
    float D = 0.0f, log_T = 0.0f, prev_log_T = 0.0f;
    float T_cur = expf(log_T);   // expf(log_T) of the termination test is the next step's transmittance
    int last_face = -1, last_tet = -1;
    bool active = false;
    uint32_t n_contrib = 0;
    int curr_face = first_face, curr_tet = first_tet;
    int4* trail = p.trail + bpix;
    const uint32_t trail_cap = (uint32_t)p.trail_cap;

    while (!done) {
        // loads of this step: shading record, intensity, adjacency record (tet 0 stands in when the ray
        // is about to leave the mesh; its result is not used)
        const float4* sh4 = reinterpret_cast<const float4*>(p.shade + curr_face);
        const float4 s0 = sh4[0], s1 = sh4[1], s2 = sh4[2];
        const float log1m = s2.z;
        const float intense = p.faces_intense[(size_t)b * p.F + curr_face];
        const TetStep s = tet_step<true, IRR>(p, b, p.tet_rec + (curr_tet >= 0 ? curr_tet : 0), curr_face, ro, rd);
        // Trail entry: face id; bit 31 flags a tet in which a second side is hit with an inward normal.
        // The reference's reverse march (backward.cu:382-477) finds two entry candidates there and gives
        // up on the ray (its error case 3), leaving this and all earlier faces without gradient; the
        // replay reproduces that.  (The side we entered through always qualifies as the first candidate:
        // it passed the same hit test one step earlier and its normal sign is checked by tet_step.)
        if (n_contrib < trail_cap)   // streaming: read once, by the backward pass
            __stcs(trail + (size_t)n_contrib * BI, make_int4(curr_face | (s.opposite ? (int)0x80000000u : 0), __float_as_int(rt),
                                                             __float_as_int(iu), __float_as_int(iv)));

        // 1. composite the current face (forward.cu:600-653)
        const float3 c0 = f3(s0.x, s0.y, s0.z), c1 = f3(s0.w, s1.x, s1.y), c2 = f3(s1.z, s1.w, s2.x);
        const float opacity = s2.y;
        float3 col = (c0 + (c1 - c0) * iu + (c2 - c0) * iv);
        col = col * intense;
        const float tmp_T = T_cur;
        C = C + tmp_T * opacity * col;
        const float pw = dep.aw + rt * dep.bw;
        float pd = (dep.az + rt * dep.bz) * (1.0f / clamp_w(pw));   // tet_depth_at
        if (fabsf(pw) < (1.0f + fabsf(pd)) * dep_scale) {            // close to the camera plane
            if (!IRR) { redo = true; break; }                         // the second pass re-marches the ray
            pd = tet_depth_exact(p.mv + 16 * b, p.proj + 16 * b, ro, rd, rt);
        }
        D += tmp_T * opacity * pd;

        prev_log_T = log_T;
        if (opacity < 1.0f) log_T += log1m;
        else log_T = logf(DMR_T_EPS * 0.1f);
        T_cur = expf(log_T);
        if (T_cur < DMR_T_EPS) { done = true; active = true; }

        n_contrib++;
        last_face = curr_face;
        last_tet = curr_tet;

        // 2. next face (forward.cu:662-775)
        if (curr_tet == -1) { active = true; done = true; }
        if (!done) {
            if (!s.ok) { done = true; if (!IRR) redo = s.irregular; }   // numerical failure: pixel stays inactive
            curr_face = s.face; curr_tet = s.tet;
            rt = s.rt; iu = s.iu; iv = s.iv;
        }
    }

    if (!IRR && redo) { p.active[bpix] = DMR_TET_REDO; return; }   // the second pass writes this pixel
    p.final_log_T[bpix] = log_T;
    p.prev_log_T[bpix] = prev_log_T;
    p.last_face[bpix] = last_face;
    p.last_tet[bpix] = last_tet;
    p.n_contrib[bpix] = n_contrib;
    p.active[bpix] = active ? 1 : 0;
    if (active) {
        float fT = T_cur;
        p.out_color[(size_t)b * 3 * HW + 0 * HW + pix] = C.x + fT * p.bg[0];
        p.out_color[(size_t)b * 3 * HW + 1 * HW + pix] = C.y + fT * p.bg[1];
        p.out_color[(size_t)b * 3 * HW + 2 * HW + pix] = C.z + fT * p.bg[2];
        p.out_depth[bpix] = D + fT * 1.0f;
        p.out_active[bpix] = 1.0f;
    } else {
        p.out_color[(size_t)b * 3 * HW + 0 * HW + pix] = p.bg[0];
        p.out_color[(size_t)b * 3 * HW + 1 * HW + pix] = p.bg[1];
        p.out_color[(size_t)b * 3 * HW + 2 * HW + pix] = p.bg[2];
        p.out_depth[bpix] = 1.0f;
        p.out_active[bpix] = 0.0f;
    }
}

int tet_march_forward(const TetParams& p, cudaStream_t stream)
{
    dim3 grid((p.W + 7) / 8, (p.H + MARCH_ROWS - 1) / MARCH_ROWS, p.B);
    ProfScope prof(ST_TET_FWD, stream);
    DMR_CUDA(dmr_launch(tet_march_fwd_kernel<false>, dim3(grid), dim3(MARCH_THREADS), 0, stream, p));
    DMR_LAUNCH_CHECK("tet_march_fwd_kernel");
    count_launch(1);   // two kernels under one scope
    DMR_CUDA(dmr_launch(tet_march_fwd_kernel<true>, dim3(grid), dim3(MARCH_THREADS), 0, stream, p));
    DMR_LAUNCH_CHECK("tet_march_fwd_kernel<irregular>");
    return 0;
}

// ---------------------------------------------------------------------------
// backward march
// ---------------------------------------------------------------------------
// Per-ray state of the reverse compositing recurrence (backward.cu:272-339).
struct TetBwdState {
    float prev_log_T, last_alpha, last_depth, accum_recd;
    float last_color[3], accum_rec[3];
    bool first_iter;
    float det_sv;       // deterministic mode: fixed-point scale (det.cuh)
    ptrdiff_t det_hi;   // ... and the offset of the high words
};

// Gradient terms of one crossed face (backward.cu:252-360) and their reduction.
// The reference issues 10 scalar atomics per crossed face (9 vertex-colour terms + opacity), which
// bounds its backward pass by the reduction rate of the LSU/L2 (measured, tools/ubench_red.cu).
// Here the nine colour terms are three 16-byte vector reductions into a float4-per-vertex accumulator
// (4.4 MB at C3, L2-resident; tet_grad_vertex_kernel folds it into dL_dverts_color[P,3]) + one scalar.
// (Also measured: one 48-byte statistics record per face + a finish kernel, as in the tri renderer --
// 0.06 ms slower at C3 because the records (152 MB) have to be zeroed, written and read back; and opportunistic
// warp aggregation of the lanes that hold the same face (match.any + one shuffle round per extra lane): no gain,
// 779 vs 770 us.)
template <bool DET>
__device__ __forceinline__ void tet_bwd_face(const TetParams& p, TetBwdState& st, int face, float rt, float iu, float iv,
                                             const float4 s0, const float4 s1, const float4 s2, const float4 s3,
                                             float intense, const TetDepth& dep,
                                             const float dLc[3], float gd, float bg_dot, float bd_dot, float final_T,
                                             float final_prev_T)
{
    const float3 c0 = f3(s0.x, s0.y, s0.z), c1 = f3(s0.w, s1.x, s1.y), c2 = f3(s1.z, s1.w, s2.x);
    const float opacity = s2.y;
    const float log1m = s2.z;

    // backward.cu:252-270
    float i0 = 1.0f - iu - iv, i1 = iu, i2 = iv;
    float3 col = (i0 * c0) + (i1 * c1) + (i2 * c2);
    col = col * intense;
    const float pd = tet_depth_at(dep, rt);

    if (!st.first_iter) st.prev_log_T = st.prev_log_T - log1m;
    st.first_iter = false;
    float prev_T = expf(st.prev_log_T);

    // backward.cu:288-339
    float dL_dcol[3];
    float dL_dopa = 0.0f;
    const float tc[3] = { col.x, col.y, col.z };
#pragma unroll
    for (int ch = 0; ch < 3; ch++) {
        const float c = tc[ch];
        st.accum_rec[ch] = st.last_alpha * st.last_color[ch] + (1.f - st.last_alpha) * st.accum_rec[ch];
        st.last_color[ch] = c;
        dL_dcol[ch] = dLc[ch] * opacity * prev_T;
        dL_dopa += (c - st.accum_rec[ch]) * dLc[ch];
    }
    st.accum_recd = st.last_alpha * st.last_depth + (1.f - st.last_alpha) * st.accum_recd;
    st.last_depth = pd;
    dL_dopa += (pd - st.accum_recd) * gd;
    dL_dopa *= prev_T;
    st.last_alpha = opacity;
    if (opacity == 1.0f) {
        dL_dopa += (-final_prev_T) * bg_dot;
        dL_dopa += (-final_prev_T) * bd_dot;
    } else {
        dL_dopa += (-final_T / (1.f - opacity)) * bg_dot;
        dL_dopa += (-final_T / (1.f - opacity)) * bd_dot;
    }

    // backward.cu:341-360
    const float g00 = i0 * dL_dcol[0] * intense, g01 = i0 * dL_dcol[1] * intense, g02 = i0 * dL_dcol[2] * intense;
    const float g10 = i1 * dL_dcol[0] * intense, g11 = i1 * dL_dcol[1] * intense, g12 = i1 * dL_dcol[2] * intense;
    const float g20 = i2 * dL_dcol[0] * intense, g21 = i2 * dL_dcol[1] * intense, g22 = i2 * dL_dcol[2] * intense;
    const int vi0 = __float_as_int(s2.w), vi1 = __float_as_int(s3.x), vi2 = __float_as_int(s3.y);
    if (DET) {
        // deterministic mode (det.cuh): 64-bit fixed-point accumulators, any arrival order gives the same bits
        const float sv = st.det_sv;
        const ptrdiff_t hi = st.det_hi;
        const uint32_t* gm = p.det_gmax;
        long long* a0 = p.det_vert + 4 * (size_t)vi0; long long* a1 = p.det_vert + 4 * (size_t)vi1; long long* a2 = p.det_vert + 4 * (size_t)vi2;
        det_add(a0 + 0, g00, sv, hi, gm); det_add(a0 + 1, g01, sv, hi, gm); det_add(a0 + 2, g02, sv, hi, gm);
        det_add(a1 + 0, g10, sv, hi, gm); det_add(a1 + 1, g11, sv, hi, gm); det_add(a1 + 2, g12, sv, hi, gm);
        det_add(a2 + 0, g20, sv, hi, gm); det_add(a2 + 1, g21, sv, hi, gm); det_add(a2 + 2, g22, sv, hi, gm);
        det_add(p.det_fopa + face, dL_dopa, sv, hi, gm);
        return;
    }
    red_add_v4(reinterpret_cast<float*>(p.grad_vacc + vi0), g00, g01, g02, 0.0f);
    red_add_v4(reinterpret_cast<float*>(p.grad_vacc + vi1), g10, g11, g12, 0.0f);
    red_add_v4(reinterpret_cast<float*>(p.grad_vacc + vi2), g20, g21, g22, 0.0f);
    atomicAdd(&p.dL_dfaces_opacity[face], dL_dopa);
}

// Camera gradients (CAM instantiations; DESIGN.md 3.4).  The camera enters a step through the ray -- (t, u, v) of the
// Moeller-Trumbore test against the face's triangle p0 p1 p2 in faces[] order -- and through the hit-point depth
// pd = Z / clamp_w(W), Z = az + t bz, W = aw + t bw, whose coefficients depend on ro, rd and the z / w rows of
// proj * mv.  A lane accumulates dL/dro and dL/drd through (t, u, v), and dL/d(az, bz, aw, bw); tet_march_bwd_cam
// chains them into the matrices after the walk.  With T = ro - p0, E1 = p1 - p0, E2 = p2 - p0, N = E2 x E1 and
// D = rd.N:  dt/dro = -N / D, dt/drd = -t N / D, du/dro = (rd x E2) / D, du/drd = (E2 x T - u N) / D,
// dv/dro = (E1 x rd) / D, dv/drd = (T x E1 - v N) / D.
struct TetCamAcc {
    float3 g_ro, g_rd;
    float g_az, g_bz, g_aw, g_bw;
};

__device__ __forceinline__ void tet_cam_step(TetCamAcc& a, const TetBwdState& st, const TetDepth& dep, float3 ro, float3 rd,
                                             float rt, float iu, float iv, const float4 s0, const float4 s1, const float4 s2,
                                             float intense, const float dLc[3], float gd, const float4 v0, const float4 v1,
                                             float v2z)
{
    const float3 c0 = f3(s0.x, s0.y, s0.z), c1 = f3(s0.w, s1.x, s1.y), c2 = f3(s1.z, s1.w, s2.x);
    const float w = s2.y * expf(st.prev_log_T);      // T_k alpha_k of the step (does not depend on the camera)
    const float3 dc1 = c1 - c0, dc2 = c2 - c0;
    const float wi = w * intense;
    const float dL_du = wi * (dLc[0] * dc1.x + dLc[1] * dc1.y + dLc[2] * dc1.z);
    const float dL_dv = wi * (dLc[0] * dc2.x + dLc[1] * dc2.y + dLc[2] * dc2.z);
    // depth: no derivative through a clamped w
    const float Z = dep.az + rt * dep.bz, Wr = dep.aw + rt * dep.bw, Wc = clamp_w(Wr);
    const float gZ = w * gd / Wc;
    const float gW = Wc == Wr ? -gZ * (Z / Wc) : 0.0f;
    a.g_az += gZ; a.g_bz += gZ * rt; a.g_aw += gW; a.g_bw += gW * rt;
    const float dL_dt = gZ * dep.bz + gW * dep.bw;
    // (t, u, v): the two rd x / x T terms of u and v share M = (dL_du E2 - dL_dv E1) / D
    const float3 p0 = f3(v0.x, v0.y, v0.z), p1 = f3(v0.w, v1.x, v1.y), p2 = f3(v1.z, v1.w, v2z);
    const float3 E1 = p1 - p0, E2 = p2 - p0, Tv = ro - p0;
    const float3 N = cross3(E2, E1);
    const float iD = 1.0f / dot3(rd, N);
    const float ku = dL_du * iD, kv = dL_dv * iD, kt = dL_dt * iD;
    const float kn = kt * rt + ku * iu + kv * iv;
    const float3 M = ku * E2 - kv * E1;
    a.g_ro = a.g_ro + cross3(rd, M) - kt * N;
    a.g_rd = a.g_rd + cross3(M, Tv) - kn * N;
}

// The sensitivities of a step as tet_cam_step forms them -- k_u = dL/du / D, k_v, k_t likewise, k_n = k_u u + k_v v + k_t t
// -- and the step's triangle, for the vertex-position instantiations (CAM: also the depth-coefficient terms into `a`).
// tet_cam_step keeps its own copy of these lines: routed through this function, the camera kernels compile to
// differently scheduled code.
struct TetStepGrad {
    float3 E1, E2, Tv, N;
    float ku, kv, kt, kn;
};

template <bool CAM>
__device__ __forceinline__ TetStepGrad tet_step_grad(TetCamAcc& a, const TetBwdState& st, const TetDepth& dep, float3 ro,
                                                     float3 rd, float rt, float iu, float iv, const float4 s0,
                                                     const float4 s1, const float4 s2, float intense, const float dLc[3],
                                                     float gd, const float4 v0, const float4 v1, float v2z)
{
    const float3 c0 = f3(s0.x, s0.y, s0.z), c1 = f3(s0.w, s1.x, s1.y), c2 = f3(s1.z, s1.w, s2.x);
    const float w = s2.y * expf(st.prev_log_T);      // T_k alpha_k of the step (does not depend on the camera)
    const float3 dc1 = c1 - c0, dc2 = c2 - c0;
    const float wi = w * intense;
    const float dL_du = wi * (dLc[0] * dc1.x + dLc[1] * dc1.y + dLc[2] * dc1.z);
    const float dL_dv = wi * (dLc[0] * dc2.x + dLc[1] * dc2.y + dLc[2] * dc2.z);
    // depth: no derivative through a clamped w
    const float Z = dep.az + rt * dep.bz, Wr = dep.aw + rt * dep.bw, Wc = clamp_w(Wr);
    const float gZ = w * gd / Wc;
    const float gW = Wc == Wr ? -gZ * (Z / Wc) : 0.0f;
    if constexpr (CAM) { a.g_az += gZ; a.g_bz += gZ * rt; a.g_aw += gW; a.g_bw += gW * rt; }
    const float dL_dt = gZ * dep.bz + gW * dep.bw;
    const float3 p0 = f3(v0.x, v0.y, v0.z), p1 = f3(v0.w, v1.x, v1.y), p2 = f3(v1.z, v1.w, v2z);
    TetStepGrad k;
    k.E1 = p1 - p0; k.E2 = p2 - p0; k.Tv = ro - p0;
    k.N = cross3(k.E2, k.E1);
    const float iD = 1.0f / dot3(rd, k.N);
    k.ku = dL_du * iD; k.kv = dL_dv * iD; k.kt = dL_dt * iD;
    k.kn = k.kt * rt + k.ku * iu + k.kv * iv;
    return k;
}

// Vertex-position gradients (VERT instantiations; DESIGN.md 3.4).  A vertex enters a step only through (t, u, v) of
// the Moeller-Trumbore test against the face's triangle p0 p1 p2 (TetFaceRec, faces[] order); colours, opacities and the
// depth coefficients do not depend on it.  With the sensitivities of tet_step_grad:
//     g_T  = k_u (rd x E2) + k_v (E1 x rd) - k_t N           (= the camera path's dL/dro of the step)
//     g_E1 = k_v (rd x T)  + k_t (E2 x T)  - k_n (rd x E2)
//     g_E2 = k_u (T x rd)  + k_t (T x E1)  - k_n (E1 x rd)
//     dL/dp0 = -g_T - g_E1 - g_E2,   dL/dp1 = g_E1,   dL/dp2 = g_E2
// scattered to the vertex ids TetShade.i0..i2 (the same vertices in the same order): three vector reductions into
// a.vg.grad_pacc, or nine fixed-point additions with the geometry scale a.det_sg into a.vg.det_pos.  CAM: the camera
// terms of tet_cam_step from the same sensitivities, into the TetCamAcc part of `a`.
struct TetVertAcc : TetCamAcc {
    TetVertGrad vg;
    float det_sg;   // deterministic mode: the fixed-point scale of positions (det.cuh)
};

template <bool DET, bool CAM>
__device__ __forceinline__ void tet_vert_step(const TetParams& p, TetVertAcc& a, const TetBwdState& st, const TetDepth& dep, float3 ro, float3 rd, float rt, float iu, float iv,
                                              const float4 s0, const float4 s1, const float4 s2, const float4 s3,
                                              float intense, const float dLc[3], float gd, const float4 v0, const float4 v1,
                                              float v2z)
{
    const TetStepGrad k = tet_step_grad<CAM>(a, st, dep, ro, rd, rt, iu, iv, s0, s1, s2, intense, dLc, gd, v0, v1, v2z);
    const float3 M = k.ku * k.E2 - k.kv * k.E1;
    if constexpr (CAM) {
        a.g_ro = a.g_ro + cross3(rd, M) - k.kt * k.N;
        a.g_rd = a.g_rd + cross3(M, k.Tv) - k.kn * k.N;
    }
    const float3 gT = cross3(rd, M) - k.kt * k.N;
    const float3 gE1 = cross3(k.kv * rd + k.kt * k.E2, k.Tv) - k.kn * cross3(rd, k.E2);
    const float3 gE2 = cross3(k.Tv, k.ku * rd + k.kt * k.E1) - k.kn * cross3(k.E1, rd);
    const float3 g0 = -(gT + gE1 + gE2);
    const int vi0 = __float_as_int(s2.w), vi1 = __float_as_int(s3.x), vi2 = __float_as_int(s3.y);
    const TetVertGrad& vg = a.vg;
    if constexpr (DET) {
        const float sg = a.det_sg;
        const ptrdiff_t hi = st.det_hi;
        const uint32_t* gm = p.det_gmax;
        long long* a0 = vg.det_pos + 4 * (size_t)vi0; long long* a1 = vg.det_pos + 4 * (size_t)vi1; long long* a2 = vg.det_pos + 4 * (size_t)vi2;
        det_add(a0 + 0, g0.x, sg, hi, gm); det_add(a0 + 1, g0.y, sg, hi, gm); det_add(a0 + 2, g0.z, sg, hi, gm);
        det_add(a1 + 0, gE1.x, sg, hi, gm); det_add(a1 + 1, gE1.y, sg, hi, gm); det_add(a1 + 2, gE1.z, sg, hi, gm);
        det_add(a2 + 0, gE2.x, sg, hi, gm); det_add(a2 + 1, gE2.y, sg, hi, gm); det_add(a2 + 2, gE2.z, sg, hi, gm);
    } else {
        red_add_v4(reinterpret_cast<float*>(vg.grad_pacc + vi0), g0.x, g0.y, g0.z, 0.0f);
        red_add_v4(reinterpret_cast<float*>(vg.grad_pacc + vi1), gE1.x, gE1.y, gE1.z, 0.0f);
        red_add_v4(reinterpret_cast<float*>(vg.grad_pacc + vi2), gE2.x, gE2.y, gE2.z, 0.0f);
    }
}

// Face-intensity gradients (INT instantiations; DESIGN.md 3.4).  The step's colour is intense * interp with
// interp = i0 c0 + i1 c1 + i2 c2, so with tet_bwd_face's dL_dcol[ch] = dLc[ch] opacity prev_T
//     dL/dfaces_intense[b, face] += sum_ch dL_dcol[ch] interp[ch]
// formed from interp itself, not col / intense: a face of intensity 0 gets its (generally nonzero) gradient.  One scalar
// reduction into ig.dL_dfint, or one fixed-point addition with the value scale into ig.det_fint.  Called after
// tet_bwd_face for the same step, whose st.prev_log_T it reads.
template <class Base>
struct TetIntAcc : Base {
    TetIntGrad ig;
};

template <bool DET>
__device__ __forceinline__ void tet_int_step(const TetParams& p, const TetIntGrad& ig, const TetBwdState& st, int b,
                                             int face, float iu, float iv, const float4 s0, const float4 s1,
                                             const float4 s2, const float dLc[3])
{
    const float3 c0 = f3(s0.x, s0.y, s0.z), c1 = f3(s0.w, s1.x, s1.y), c2 = f3(s1.z, s1.w, s2.x);
    const float opacity = s2.y;
    const float i0 = 1.0f - iu - iv;
    const float3 interp = (i0 * c0) + (iu * c1) + (iv * c2);
    const float prev_T = expf(st.prev_log_T);
    const float g = dLc[0] * opacity * prev_T * interp.x + dLc[1] * opacity * prev_T * interp.y +
                    dLc[2] * opacity * prev_T * interp.z;
    const size_t i = (size_t)b * p.F + face;
    if constexpr (DET) det_add(ig.det_fint + i, g, st.det_sv, ig.det_hi, p.det_gmax);
    else atomicAdd(ig.dL_dfint + i, g);
}

// Backward march.  Steps recorded in the face trail (all of them unless a ray composited more than
// trail_cap faces) are replayed in reverse: face id and the forward pass's own (t,u,v) from the trail
// (one coalesced 16-byte load), all loads independent of the previous step and issued one step ahead.  Steps beyond the cap are re-marched through the adjacency records exactly like
// the reference (backward.cu:382-477) until the recorded part is reached.
// (Measured and rejected: the replay alone in its own kernel -- rays beyond the cap left to a second launch -- so that
// it fits 80 / 72 / 64 registers and 12 / 14 / 16 CTAs per SM instead of 10: C3 588.6 / 601 / 652 us against 587.8 us.
// More resident warps do not help: the kernel is bound by the wavefronts its per-lane gathers and reductions push
// through the L1 data pipe, not by the latency of a single chain.)
// CAM: also accumulate the camera terms of every walked step into `cam` (tet_cam_step); the face's vertices are loaded
// with its shading record.  The early returns end the walk only: tet_march_bwd_cam reduces after it on every lane.
// VERT: also scatter the vertex-position terms of every walked step (tet_vert_step, sharing the triangle and the
// sensitivities with CAM); `cam` is then a TetVertAcc.
// INT: also add the face-intensity term of every walked step (tet_int_step); `cam` is then a TetIntAcc<...>.
// ALPHA: the image also has an alpha cotangent dL_dalpha [B,H,W] (alpha = 1 - expf(final_log_T) on active pixels, the
// factor the forward pass multiplies the background by; DESIGN.md 3.4): it enters where the background term does, as
// bd_dot - dL_dalpha, so tet_bwd_face is unchanged.
template <bool DET, bool CAM, bool VERT = false, bool INT = false, class Acc = TetCamAcc, bool ALPHA = false>
__device__ __forceinline__ void tet_march_bwd_body(const TetParams& p, Acc& cam, const float* __restrict__ dL_dalpha = nullptr)
{
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int b = blockIdx.z;
    const uint32_t px = blockIdx.x * 8 + (lane & 7);
    const uint32_t py = blockIdx.y * MARCH_ROWS + warp * 4 + (lane >> 3);
    if (!(px < (uint32_t)p.W && py < (uint32_t)p.H)) return;
    const size_t HW = (size_t)p.W * p.H;
    const size_t BI = (size_t)p.B * HW;
    const size_t pix = (size_t)py * p.W + px;
    const size_t bpix = (size_t)b * HW + pix;

    if (!p.active[bpix]) return;                    // backward.cu:160-163
    const int last_face = p.last_face[bpix];
    if (last_face == -1) return;                    // backward.cu:190-193
    const int last_tet = p.last_tet[bpix];
    const int first_face = p.first_face[bpix];
    int k = (int)p.n_contrib[bpix] - 1;             // index of the step to process next, counting down

    const float fin_prev_log_T = p.prev_log_T[bpix];
    const float fin_log_T = p.final_log_T[bpix];
    const float final_prev_T = expf(fin_prev_log_T);
    const float final_T = expf(fin_log_T);

    const float g0 = p.dL_dcolor[(size_t)b * 3 * HW + 0 * HW + pix];
    const float g1 = p.dL_dcolor[(size_t)b * 3 * HW + 1 * HW + pix];
    const float g2 = p.dL_dcolor[(size_t)b * 3 * HW + 2 * HW + pix];
    const float gd = p.dL_ddepth[bpix];
    const float dLc[3] = { g0, g1, g2 };

    float3 ro, rd;
    tet_pixel_ray(p, b, px, py, bpix, ro, rd);
    const TetDepth dep = tet_depth_setup(p.mv + 16 * b, p.proj + 16 * b, ro, rd);

    // backward.cu:324-329
    float bg_dot = 0; bg_dot += p.bg[0] * g0; bg_dot += p.bg[1] * g1; bg_dot += p.bg[2] * g2;
    float bd_dot = 0; bd_dot += 1.0 * gd;
    if constexpr (ALPHA) bd_dot -= dL_dalpha[bpix];

    TetBwdState st;
    st.det_sv = 0.0f;
    st.det_hi = 0;
    if (DET) {
        float sg;
        det_scales(*p.det_gmax, st.det_sv, sg);
        if constexpr (VERT) cam.det_sg = sg;
        st.det_hi = TetDetLayout::hi_offset(p.P, p.F);
    }
    st.prev_log_T = fin_prev_log_T;
    st.last_alpha = 0.0f; st.last_depth = 0.0f; st.accum_recd = 0.0f;
#pragma unroll
    for (int ch = 0; ch < 3; ch++) { st.last_color[ch] = 0.0f; st.accum_rec[ch] = 0.0f; }
    st.first_iter = true;

    // ---- part 1 (rare): steps beyond the trail, re-marched through the adjacency records
    if (k >= p.trail_cap) {
        float rt, iu, iv;
        {
            const float* w = reinterpret_cast<const float*>(p.face_rec + (size_t)b * p.F + last_face);
            float3 tuv = f3(0, 0, 0);
            ray_tri_hit(ro, rd, f3(w[0], w[1], w[2]), f3(w[3], w[4], w[5]), f3(w[6], w[7], w[8]), tuv);
            rt = tuv.x; iu = tuv.y; iv = tuv.z;
        }
        int curr_face = last_face, curr_tet = last_tet;
        // the tet on the near side of the last face: backward.cu:224-232
        {
            const TetShade* sh = p.shade + curr_face;
            const int cand[2] = { sh->t0, sh->t1 };
            for (int i = 0; i < 2; i++) {
                if (cand[i] == curr_tet) continue;
                curr_tet = cand[i];
                break;
            }
        }
        while (k >= p.trail_cap) {
            const float4* sh4 = reinterpret_cast<const float4*>(p.shade + curr_face);
            const float4 s0 = sh4[0], s1 = sh4[1], s2 = sh4[2], s3 = sh4[3];
            const float intense = p.faces_intense[(size_t)b * p.F + curr_face];
            float4 v0, v1;
            float v2z;
            if constexpr (CAM || VERT) {
                const float4* fr = reinterpret_cast<const float4*>(p.face_rec + (size_t)b * p.F + curr_face);
                v0 = fr[0]; v1 = fr[1]; v2z = reinterpret_cast<const float*>(fr)[8];
            }
            tet_bwd_face<DET>(p, st, curr_face, rt, iu, iv, s0, s1, s2, s3, intense, dep, dLc, gd, bg_dot, bd_dot,
                         final_T, final_prev_T);
            // (t, u, v) of the re-march: recomputed, the same bits as the forward march's
            if constexpr (VERT)
                tet_vert_step<DET, CAM>(p, cam, st, dep, ro, rd, rt, iu, iv, s0, s1, s2, s3, intense, dLc, gd, v0, v1, v2z);
            else if constexpr (CAM)
                tet_cam_step(cam, st, dep, ro, rd, rt, iu, iv, s0, s1, s2, intense, dLc, gd, v0, v1, v2z);
            if constexpr (INT) tet_int_step<DET>(p, cam.ig, st, b, curr_face, iu, iv, s0, s1, s2, dLc);
            k--;
            if (curr_face == first_face) return;         // backward.cu:363-366
            if (curr_tet == -1) return;                  // backward.cu:373-376
            TetStep s = tet_step<false, true>(p, b, p.tet_rec + curr_tet, curr_face, ro, rd);
            if (!s.ok) return;
            curr_face = s.face; curr_tet = s.tet;
            rt = s.rt; iu = s.iu; iv = s.iv;
        }
    }

    // ---- part 2: replay the trail in reverse, loads one step ahead
    const int4* trail = p.trail + bpix;
    const float* fint = p.faces_intense + (size_t)b * p.F;

    int4 e = __ldcs(trail + (size_t)k * BI);
    int4 e_next = k > 0 ? __ldcs(trail + (size_t)(k - 1) * BI) : make_int4(0, 0, 0, 0);
    int face = e.x & 0x7fffffff;
    float4 s0, s1, s2, s3;
    float intense;
    {
        const float4* sh4 = reinterpret_cast<const float4*>(p.shade + face);
        s0 = sh4[0]; s1 = sh4[1]; s2 = sh4[2]; s3 = sh4[3];
        intense = fint[face];
    }
    // CAM, VERT: the face's triangle (TetFaceRec p0 p1 p2), loaded together with the shading record
    const float4* frec = reinterpret_cast<const float4*>(p.face_rec + (size_t)b * p.F);
    float4 v0, v1;
    float v2z;
    if constexpr (CAM || VERT) { v0 = frec[4 * face]; v1 = frec[4 * face + 1]; v2z = reinterpret_cast<const float*>(frec + 4 * face)[8]; }
    for (; k >= 0; k--) {
        // issue the loads of step k-1 (face id known since the previous iteration), then work on step k
        const int nf = e_next.x & 0x7fffffff;
        const bool stop_here = e_next.x < 0;   // the reference's reverse march fails between step k and k-1
        const float4* sh4 = reinterpret_cast<const float4*>(p.shade + nf);
        const float4 ns0 = sh4[0], ns1 = sh4[1], ns2 = sh4[2], ns3 = sh4[3];
        const float nint = fint[nf];
        float4 nv0, nv1;
        float nv2z;
        if constexpr (CAM || VERT) { nv0 = frec[4 * nf]; nv1 = frec[4 * nf + 1]; nv2z = reinterpret_cast<const float*>(frec + 4 * nf)[8]; }
        const int4 e_cur = e;
        e = e_next;
        e_next = k > 1 ? __ldcs(trail + (size_t)(k - 2) * BI) : make_int4(0, 0, 0, 0);

        // (t, u, v) of the step: the forward march's own values
        tet_bwd_face<DET>(p, st, face, __int_as_float(e_cur.y), __int_as_float(e_cur.z), __int_as_float(e_cur.w), s0, s1, s2, s3,
                          intense, dep, dLc, gd, bg_dot, bd_dot, final_T, final_prev_T);
        if constexpr (VERT)
            tet_vert_step<DET, CAM>(p, cam, st, dep, ro, rd, __int_as_float(e_cur.y), __int_as_float(e_cur.z),
                                    __int_as_float(e_cur.w), s0, s1, s2, s3, intense, dLc, gd, v0, v1, v2z);
        else if constexpr (CAM)
            tet_cam_step(cam, st, dep, ro, rd, __int_as_float(e_cur.y), __int_as_float(e_cur.z), __int_as_float(e_cur.w), s0, s1,
                         s2, intense, dLc, gd, v0, v1, v2z);
        if constexpr (INT)
            tet_int_step<DET>(p, cam.ig, st, b, face, __int_as_float(e_cur.z), __int_as_float(e_cur.w), s0, s1, s2, dLc);

        if (stop_here) break;
        face = nf;
        s0 = ns0; s1 = ns1; s2 = ns2; s3 = ns3;
        intense = nint;
        if constexpr (CAM || VERT) { v0 = nv0; v1 = nv1; v2z = nv2z; }
    }
}

// Once per vertex: float4 accumulator -> dL_dverts_color[P,3].
__global__ void __launch_bounds__(MARCH_THREADS) tet_march_bwd_kernel(TetParams p)
{
    griddep_wait();
    TetCamAcc unused;
    tet_march_bwd_body<false, false>(p, unused);
}
__global__ void __launch_bounds__(MARCH_THREADS) tet_march_bwd_det_kernel(TetParams p)
{
    griddep_wait();
    TetCamAcc unused;
    tet_march_bwd_body<true, false>(p, unused);
}
// Vertex-position instantiations: position gradients into vg.grad_pacc (tet_grad_position_kernel folds them into
// vg.dL_dverts) or vg.det_pos (tet_det_convert_position_kernel).
__global__ void __launch_bounds__(MARCH_THREADS) tet_march_bwd_vert_kernel(TetParams p, TetVertGrad vg)
{
    griddep_wait();
    TetVertAcc a;
    a.vg = vg;
    tet_march_bwd_body<false, false, true>(p, a);
}
__global__ void __launch_bounds__(MARCH_THREADS) tet_march_bwd_vert_det_kernel(TetParams p, TetVertGrad vg)
{
    griddep_wait();
    TetVertAcc a;
    a.vg = vg;
    tet_march_bwd_body<true, false, true>(p, a);
}
// Face-intensity instantiations: dL/dfaces_intense straight into ig.dL_dfint, or into ig.det_fint
// (tet_det_convert_intensity_kernel); with or without the vertex-position terms.
__global__ void __launch_bounds__(MARCH_THREADS) tet_march_bwd_int_kernel(TetParams p, TetIntGrad ig)
{
    griddep_wait();
    TetIntAcc<TetCamAcc> a;
    a.ig = ig;
    tet_march_bwd_body<false, false, false, true>(p, a);
}
__global__ void __launch_bounds__(MARCH_THREADS) tet_march_bwd_int_det_kernel(TetParams p, TetIntGrad ig)
{
    griddep_wait();
    TetIntAcc<TetCamAcc> a;
    a.ig = ig;
    tet_march_bwd_body<true, false, false, true>(p, a);
}
__global__ void __launch_bounds__(MARCH_THREADS) tet_march_bwd_vert_int_kernel(TetParams p, TetVertGrad vg, TetIntGrad ig)
{
    griddep_wait();
    TetIntAcc<TetVertAcc> a;
    a.vg = vg;
    a.ig = ig;
    tet_march_bwd_body<false, false, true, true>(p, a);
}
__global__ void __launch_bounds__(MARCH_THREADS) tet_march_bwd_vert_int_det_kernel(TetParams p, TetVertGrad vg, TetIntGrad ig)
{
    griddep_wait();
    TetIntAcc<TetVertAcc> a;
    a.vg = vg;
    a.ig = ig;
    tet_march_bwd_body<true, false, true, true>(p, a);
}

// Camera-gradient instantiations: the walk of tet_march_bwd_body<DET, true>, then per lane the chain of its pixel into
// the matrices, and one record of DMR_TET_CAM_REC floats per (view, CTA), summed in a fixed order (no float atomics:
// reproducible in both modes).  Every CTA stores its record, zeros included, so the record array is not cleared.
//   [3j + i]       dL/dinv_mv[4j + i]   = g_d[i] pv[j]           (i, j < 3)   d = L pv, L = the linear part of inv_mv
//   [9 + i]        dL/dinv_mv[12 + i]   = g_ro[i]
//   [12 + 3k + j]  dL/dinv_proj[4k + j] = (L^T g_d)[j] n[k]      (j < 3, k < 4), n = (nx, ny, -1, 1)
//   [24 + k]       dL/drz[k],  [28 + k]  dL/drw[k]               z / w rows of proj * mv (tet_depth_rows)
// tet_camera_finish_kernel applies the inverses and the direct depth-row terms.
static_assert(MARCH_THREADS == 64 && MARCH_ROWS == 8, "tet_cam_records (tet.cuh) counts 8 x 8-pixel march CTAs");
static_assert(DMR_TET_CAM_REC == 32, "one record slot per lane");
// VERT: Acc = TetVertAcc with its vg set by the caller.  INT: Acc = TetIntAcc<...> with its ig set by the caller.
template <bool DET, bool VERT = false, bool INT = false, class Acc = TetCamAcc, bool ALPHA = false>
__device__ __forceinline__ void tet_march_bwd_cam(const TetParams& p, float* __restrict__ cam_rec, Acc& a,
                                                  const float* __restrict__ dL_dalpha = nullptr)
{
    a.g_ro = f3(0, 0, 0); a.g_rd = f3(0, 0, 0);
    a.g_az = 0.0f; a.g_bz = 0.0f; a.g_aw = 0.0f; a.g_bw = 0.0f;
    tet_march_bwd_body<DET, true, VERT, INT, Acc, ALPHA>(p, a, dL_dalpha);

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int b = blockIdx.z;
    const uint32_t px = blockIdx.x * 8 + (lane & 7);
    const uint32_t py = blockIdx.y * MARCH_ROWS + warp * 4 + (lane >> 3);
    float g[DMR_TET_CAM_REC];
#pragma unroll
    for (int k = 0; k < DMR_TET_CAM_REC; k++) g[k] = 0.0f;
    if (px < (uint32_t)p.W && py < (uint32_t)p.H) {   // inactive pixels: the accumulators are zero
        const size_t bpix = (size_t)b * p.W * p.H + (size_t)py * p.W + px;
        float fx = px + 0.5f, fy = py + 0.5f;
        if (p.jitter) { const float2 j = p.jitter[bpix]; fx = j.x; fy = j.y; }   // constants: no gradient through the jitter
        const float* imv = p.inv_mv + 16 * b;
        const float* ipj = p.inv_proj + 16 * b;
        // the ray as pixel_ray<TET> forms it, with the branch of its length clamp
        const float n[4] = { pix2ndc(fx, p.W), pix2ndc(fy, p.H), -1.0f, 1.0f };
        const float3 ro = f3(imv[12], imv[13], imv[14]);
        const float4 pv4 = xform44(f3(n[0], n[1], -1.0f), ipj);
        const float4 pw = xform44(f3(pv4.x, pv4.y, pv4.z), imv);
        const float3 dv = f3(pw.x, pw.y, pw.z) - ro;
        const float len = sqrtf(dot3(dv, dv));
        const float3 rd = dv / fmaxf(len, 0.0001f);
        float rz[4], rw[4];
        tet_depth_rows(p.mv + 16 * b, p.proj + 16 * b, rz, rw);
        const float3 g_ro = a.g_ro + a.g_az * f3(rz[0], rz[1], rz[2]) + a.g_aw * f3(rw[0], rw[1], rw[2]);
        const float3 g_rd = a.g_rd + a.g_bz * f3(rz[0], rz[1], rz[2]) + a.g_bw * f3(rw[0], rw[1], rw[2]);
        // rd = d / max(|d|, 1e-4)
        const float3 gdv = len >= 0.0001f ? (g_rd - rd * dot3(rd, g_rd)) / len : g_rd / 0.0001f;
        const float pv[3] = { pv4.x, pv4.y, pv4.z };
        const float gd[3] = { gdv.x, gdv.y, gdv.z };
#pragma unroll
        for (int j = 0; j < 3; j++) {
#pragma unroll
            for (int i = 0; i < 3; i++) g[3 * j + i] = gd[i] * pv[j];
            const float lg = imv[4 * j] * gd[0] + imv[4 * j + 1] * gd[1] + imv[4 * j + 2] * gd[2];
#pragma unroll
            for (int k = 0; k < 4; k++) g[12 + 3 * k + j] = lg * n[k];
        }
        g[9] = g_ro.x; g[10] = g_ro.y; g[11] = g_ro.z;
        const float rov[3] = { ro.x, ro.y, ro.z }, rdv[3] = { rd.x, rd.y, rd.z };
#pragma unroll
        for (int k = 0; k < 3; k++) {
            g[24 + k] = a.g_az * rov[k] + a.g_bz * rdv[k];
            g[28 + k] = a.g_aw * rov[k] + a.g_bw * rdv[k];
        }
        g[27] = a.g_az; g[31] = a.g_aw;
    }
    // fixed-order reduction: warp butterfly, then the two warp sums in warp order
#pragma unroll
    for (int k = 0; k < DMR_TET_CAM_REC; k++) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) g[k] += __shfl_xor_sync(0xffffffffu, g[k], o);
    }
    __shared__ float s_cam[MARCH_THREADS];
    float x = g[0];
#pragma unroll
    for (int k = 1; k < DMR_TET_CAM_REC; k++) x = lane == k ? g[k] : x;
    s_cam[tid] = x;
    __syncthreads();
    if (tid < DMR_TET_CAM_REC)
        cam_rec[(((size_t)b * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x) * DMR_TET_CAM_REC + tid] =
            s_cam[tid] + s_cam[DMR_TET_CAM_REC + tid];
}

__global__ void __launch_bounds__(MARCH_THREADS) tet_march_bwd_cam_kernel(TetParams p, float* cam_rec)
{
    griddep_wait();
    TetCamAcc a;
    tet_march_bwd_cam<false>(p, cam_rec, a);
}
__global__ void __launch_bounds__(MARCH_THREADS) tet_march_bwd_cam_det_kernel(TetParams p, float* cam_rec)
{
    griddep_wait();
    TetCamAcc a;
    tet_march_bwd_cam<true>(p, cam_rec, a);
}
__global__ void __launch_bounds__(MARCH_THREADS) tet_march_bwd_cam_vert_kernel(TetParams p, float* cam_rec, TetVertGrad vg)
{
    griddep_wait();
    TetVertAcc a;
    a.vg = vg;
    tet_march_bwd_cam<false, true>(p, cam_rec, a);
}
__global__ void __launch_bounds__(MARCH_THREADS) tet_march_bwd_cam_vert_det_kernel(TetParams p, float* cam_rec, TetVertGrad vg)
{
    griddep_wait();
    TetVertAcc a;
    a.vg = vg;
    tet_march_bwd_cam<true, true>(p, cam_rec, a);
}
__global__ void __launch_bounds__(MARCH_THREADS) tet_march_bwd_cam_int_kernel(TetParams p, float* cam_rec, TetIntGrad ig)
{
    griddep_wait();
    TetIntAcc<TetCamAcc> a;
    a.ig = ig;
    tet_march_bwd_cam<false, false, true>(p, cam_rec, a);
}
__global__ void __launch_bounds__(MARCH_THREADS) tet_march_bwd_cam_int_det_kernel(TetParams p, float* cam_rec, TetIntGrad ig)
{
    griddep_wait();
    TetIntAcc<TetCamAcc> a;
    a.ig = ig;
    tet_march_bwd_cam<true, false, true>(p, cam_rec, a);
}
__global__ void __launch_bounds__(MARCH_THREADS) tet_march_bwd_cam_vert_int_kernel(TetParams p, float* cam_rec, TetVertGrad vg,
                                                                                   TetIntGrad ig)
{
    griddep_wait();
    TetIntAcc<TetVertAcc> a;
    a.vg = vg;
    a.ig = ig;
    tet_march_bwd_cam<false, true, true>(p, cam_rec, a);
}
__global__ void __launch_bounds__(MARCH_THREADS) tet_march_bwd_cam_vert_int_det_kernel(TetParams p, float* cam_rec,
                                                                                       TetVertGrad vg, TetIntGrad ig)
{
    griddep_wait();
    TetIntAcc<TetVertAcc> a;
    a.vg = vg;
    a.ig = ig;
    tet_march_bwd_cam<true, true, true>(p, cam_rec, a);
}

// Alpha-cotangent instantiations: the sixteen kernels above (default / deterministic x camera x vertex x intensity)
// plus dL/dalpha, which travels as an argument of its own so that TetParams stays as it is.  The accumulator type is
// the one the kernel each stands in for uses; -Xptxas -v of all of them in DESIGN.md 3.4.
template <bool VERT, bool INT>
using TetAlphaAcc = std::conditional_t<INT, TetIntAcc<std::conditional_t<VERT, TetVertAcc, TetCamAcc>>,
                                       std::conditional_t<VERT, TetVertAcc, TetCamAcc>>;
template <bool DET, bool CAM, bool VERT, bool INT>
__global__ void __launch_bounds__(MARCH_THREADS) tet_march_bwd_alpha_kernel(TetParams p, float* cam_rec, TetVertGrad vg,
                                                                            TetIntGrad ig, const float* __restrict__ dL_dalpha)
{
    griddep_wait();
    TetAlphaAcc<VERT, INT> a;
    if constexpr (VERT) a.vg = vg;
    if constexpr (INT) a.ig = ig;
    if constexpr (CAM) tet_march_bwd_cam<DET, VERT, INT, TetAlphaAcc<VERT, INT>, true>(p, cam_rec, a, dL_dalpha);
    else tet_march_bwd_body<DET, false, VERT, INT, TetAlphaAcc<VERT, INT>, true>(p, a, dL_dalpha);
}

template <bool DET>
static cudaError_t launch_tet_bwd_alpha(const TetParams& p, cudaStream_t stream, dim3 grid, float* cam_rec,
                                        const TetVertGrad* vert, const TetIntGrad* fint, const float* dL_dalpha)
{
    const TetVertGrad vg = vert ? *vert : TetVertGrad{};
    const TetIntGrad ig = fint ? *fint : TetIntGrad{};
    void (*k)(TetParams, float*, TetVertGrad, TetIntGrad, const float*);
    switch ((cam_rec ? 1 : 0) | (vert ? 2 : 0) | (fint ? 4 : 0)) {
        case 0: k = tet_march_bwd_alpha_kernel<DET, false, false, false>; break;
        case 1: k = tet_march_bwd_alpha_kernel<DET, true, false, false>; break;
        case 2: k = tet_march_bwd_alpha_kernel<DET, false, true, false>; break;
        case 3: k = tet_march_bwd_alpha_kernel<DET, true, true, false>; break;
        case 4: k = tet_march_bwd_alpha_kernel<DET, false, false, true>; break;
        case 5: k = tet_march_bwd_alpha_kernel<DET, true, false, true>; break;
        case 6: k = tet_march_bwd_alpha_kernel<DET, false, true, true>; break;
        default: k = tet_march_bwd_alpha_kernel<DET, true, true, true>; break;
    }
    return dmr_launch(k, grid, dim3(MARCH_THREADS), 0, stream, p, cam_rec, vg, ig, dL_dalpha);
}

// Face visibility statistics of a forward call (dmr_tet_face_weights; DESIGN.md 3.4), after the forward march: one
// thread per pixel, active pixels only (an inactive pixel shows the background and has alpha 0).  Every composited
// step adds its blending weight expf(log_T) * opacity -- the factor the forward march multiplies the step's colour by
// -- and 1 to the (view, face) accumulators.  Not in the march itself: its first pass hands rays through irregular
// tets to a second launch that re-marches them from the first face, and it does not know yet whether a pixel ends
// inactive.  The steps of the trail are walked forward with the march's own recurrence for log_T, and the steps of a
// ray longer than the trail are marched again from its last recorded step with the march's own exit search
// (tet_step<EXIT>), so every weight is the forward's bits.
__global__ void __launch_bounds__(MARCH_THREADS) tet_face_weights_kernel(TetParams p, FaceWeightAcc fw)
{
    griddep_wait();
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int b = blockIdx.z;
    const uint32_t px = blockIdx.x * 8 + (lane & 7);
    const uint32_t py = blockIdx.y * MARCH_ROWS + warp * 4 + (lane >> 3);
    if (!(px < (uint32_t)p.W && py < (uint32_t)p.H)) return;
    const size_t HW = (size_t)p.W * p.H;
    const size_t BI = (size_t)p.B * HW;
    const size_t bpix = (size_t)b * HW + (size_t)py * p.W + px;
    if (!p.active[bpix]) return;
    const int n = (int)p.n_contrib[bpix];
    const size_t fbase = (size_t)b * p.F;

    // steps 0 .. min(n, cap) - 1 from the trail, tet_march_fwd_kernel's arithmetic; curr_tet follows the march (the tet
    // behind face k is the first entry of face_tets[face k] that is neither the previous tet nor -1, as TetRec.next)
    const int nt = min(n, p.trail_cap);
    const int4* trail = p.trail + bpix;
    float log_T = 0.0f;
    int curr_face = -1, curr_tet = p.first_tet[bpix];
    for (int k = 0; k < nt; k++) {
        curr_face = trail[(size_t)k * BI].x & 0x7fffffff;
        const float4* sh4 = reinterpret_cast<const float4*>(p.shade + curr_face);
        const float4 s2 = sh4[2];   // (c2.z, opacity, log1m, i0)
        if (k > 0 && n > nt) {
            const int4 s3 = reinterpret_cast<const int4*>(sh4)[3];   // (i1, i2, t0, t1)
            curr_tet = (s3.z != curr_tet && s3.z != -1) ? s3.z : (s3.w != curr_tet && s3.w != -1) ? s3.w : -1;
        }
        const float opacity = s2.y;
        face_weight_add(fw, fbase + curr_face, expf(log_T) * opacity);
        if (opacity < 1.0f) log_T += s2.z;
        else log_T = logf(DMR_T_EPS * 0.1f);
    }
    // steps beyond the trail: marched again from the last recorded one with the march's own exit search (irregular
    // tets included, as its second pass), same recurrence
    if (n > nt) {
        float3 ro, rd;
        tet_pixel_ray(p, b, px, py, bpix, ro, rd);
        for (int k = nt; k < n && curr_tet >= 0; k++) {
            const TetStep s = tet_step<true, true>(p, b, p.tet_rec + curr_tet, curr_face, ro, rd);
            curr_face = s.face; curr_tet = s.tet;
            const float4 s2 = reinterpret_cast<const float4*>(p.shade + curr_face)[2];
            const float opacity = s2.y;
            face_weight_add(fw, fbase + curr_face, expf(log_T) * opacity);
            if (opacity < 1.0f) log_T += s2.z;
            else log_T = logf(DMR_T_EPS * 0.1f);
        }
    }
}

int tet_face_weights(const TetParams& p, const FaceWeightAcc& fw, float* face_weights, int* face_hits, cudaStream_t stream)
{
    dim3 grid((p.W + 7) / 8, (p.H + MARCH_ROWS - 1) / MARCH_ROWS, p.B);
    ProfScope prof(ST_TET_FACE_WEIGHTS, stream);
    count_launch(1);   // two kernels under one scope
    DMR_CUDA(dmr_launch(tet_face_weights_kernel, grid, dim3(MARCH_THREADS), 0, stream, p, fw));
    DMR_LAUNCH_CHECK("tet_face_weights_kernel");
    return face_weights_convert(p.B, p.F, fw, face_weights, face_hits, stream);
}

// One CTA per view: the view's records (tet_march_bwd_cam) are summed in a fixed order -- thread t owns component
// t % 32 of every eighth record (coalesced reads of the flat record array), then the eight partial sums of a component
// are added in thread order -- and chained into the matrices: through the inverses, dL/dA = -A^-T (dL/dA^-1) A^-T,
// plus the direct terms of the depth rows rz[k] = sum_r pj[2 + 4r] mv[4k + r] (+ pj[14] for k = 3), rw likewise with
// pj[3 + 4r] and pj[15].  The result is ADDED to dL_dmv[b] / dL_dproj[b]; this CTA is the only writer of view b.
__global__ void __launch_bounds__(256) tet_camera_finish_kernel(int nrec, const float* __restrict__ cam_rec,
                                                                const float* __restrict__ mv, const float* __restrict__ pj,
                                                                const float* __restrict__ inv_mv, const float* __restrict__ inv_proj,
                                                                float* __restrict__ dL_dmv, float* __restrict__ dL_dproj)
{
    griddep_wait();   // programmatic dependent launch: see dmr_launch (common.cuh)
    __shared__ float s_part[256];
    __shared__ float s_g[2][16];      // dL/dinv_mv, dL/dinv_proj (column-major, zeros where the forward reads nothing)
    __shared__ float s_r[8];          // dL/drz[0..3], dL/drw[0..3]
    const int b = blockIdx.x, t = threadIdx.x;
    const float* rec = cam_rec + (size_t)b * nrec * DMR_TET_CAM_REC;
    const size_t n = (size_t)nrec * DMR_TET_CAM_REC;
    float acc = 0.0f;
    for (size_t i = t; i < n; i += 256) acc += rec[i];
    s_part[t] = acc;
    __syncthreads();
    if (t < 32) {
        s_g[t >> 4][t & 15] = 0.0f;
        __syncwarp();
        float sum = 0.0f;
#pragma unroll
        for (int k = 0; k < 8; k++) sum += s_part[t + DMR_TET_CAM_REC * k];
        if (t < 9) s_g[0][4 * (t / 3) + t % 3] = sum;
        else if (t < 12) s_g[0][12 + t - 9] = sum;
        else if (t < 24) s_g[1][4 * ((t - 12) / 3) + (t - 12) % 3] = sum;
        else s_r[t - 24] = sum;
        __syncwarp();
        // thread e: entry (i, j) = (e & 3, e >> 2) of matrix t >> 4; M(r, c) = m[4c + r]
        const int m = t >> 4, e = t & 15, i = e & 3, j = e >> 2;
        const float* N = (m == 0 ? inv_mv : inv_proj) + 16 * b;
        float out = -inverse_chain(N, s_g[m], i, j);
        const float* mvb = mv + 16 * b;
        const float* pjb = pj + 16 * b;
        if (m == 0) {
            if (i < 3) out += s_r[j] * pjb[2 + 4 * i] + s_r[4 + j] * pjb[3 + 4 * i];
        } else if (i >= 2) {
            const float* R = s_r + 4 * (i - 2);
            out += j < 3 ? R[0] * mvb[j] + R[1] * mvb[4 + j] + R[2] * mvb[8 + j] + R[3] * mvb[12 + j] : R[3];
        }
        float* dst = (m == 0 ? dL_dmv : dL_dproj) + 16 * b + e;
        *dst += out;
    }
}

// Deterministic mode, last step: fixed-point accumulators -> += into dL_dverts_color[P,3] and dL_dfaces_opacity[F].
__global__ void __launch_bounds__(256) tet_det_convert_kernel(TetParams p)
{
    griddep_wait();   // programmatic dependent launch: see dmr_launch (common.cuh)
    float sv, sg;
    det_scales(*p.det_gmax, sv, sg);
    size_t i = (size_t)blockIdx.x * 256 + threadIdx.x;
    if (det_poisoned(p.det_gmax)) {
        const float nan = __int_as_float(0x7fc00000);
        if (i < (size_t)p.P) { for (int c = 0; c < 3; c++) p.dL_dverts_color[3 * i + c] = nan; }
        else if (i - (size_t)p.P < (size_t)p.F) p.dL_dfaces_opacity[i - (size_t)p.P] = nan;
        return;
    }
    if (sv == 0.0f) return;
    const double iv = 1.0 / (double)sv;
    const ptrdiff_t hi = TetDetLayout::hi_offset(p.P, p.F);
    if (i < (size_t)p.P) {
        const long long* a = p.det_vert + 4 * i;
#pragma unroll
        for (int c = 0; c < 3; c++) {
            if (det_nonzero(a + c, hi)) p.dL_dverts_color[3 * i + c] += (float)det_value(a + c, hi, iv);
        }
        return;
    }
    i -= (size_t)p.P;
    if (i < (size_t)p.F) {
        const long long* a = p.det_fopa + i;
        if (det_nonzero(a, hi)) p.dL_dfaces_opacity[i] += (float)det_value(a, hi, iv);
    }
}

__global__ void __launch_bounds__(256) tet_grad_vertex_kernel(TetParams p)
{
    griddep_wait();   // programmatic dependent launch: see dmr_launch (common.cuh)
    const int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= p.P) return;
    const float4 a = p.grad_vacc[v];
    float* o = p.dL_dverts_color + 3 * (size_t)v;
    o[0] += a.x; o[1] += a.y; o[2] += a.z;
}

// Vertex-position gradients, last step of either mode: += into dL_dverts[P,3].  The deterministic one follows the
// poisoning rule of det.cuh, as tet_det_convert_kernel does for the other gradients of the call.
__global__ void __launch_bounds__(256) tet_grad_position_kernel(int P, TetVertGrad vg)
{
    griddep_wait();   // programmatic dependent launch: see dmr_launch (common.cuh)
    const int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= P) return;
    const float4 a = vg.grad_pacc[v];
    float* o = vg.dL_dverts + 3 * (size_t)v;
    o[0] += a.x; o[1] += a.y; o[2] += a.z;
}

__global__ void __launch_bounds__(256) tet_det_convert_position_kernel(int P, int F, const uint32_t* __restrict__ gmax,
                                                                       TetVertGrad vg)
{
    griddep_wait();   // programmatic dependent launch: see dmr_launch (common.cuh)
    const size_t i = (size_t)blockIdx.x * 256 + threadIdx.x;
    if (i >= (size_t)P) return;
    if (det_poisoned(gmax)) {
        const float nan = __int_as_float(0x7fc00000);
        for (int c = 0; c < 3; c++) vg.dL_dverts[3 * i + c] = nan;
        return;
    }
    float sv, sg;
    det_scales(*gmax, sv, sg);
    if (sg == 0.0f) return;
    const double ig = 1.0 / (double)sg;
    const ptrdiff_t hi = TetDetLayout::hi_offset(P, F);
    const long long* a = vg.det_pos + 4 * i;
#pragma unroll
    for (int c = 0; c < 3; c++) {
        if (det_nonzero(a + c, hi)) vg.dL_dverts[3 * i + c] += (float)det_value(a + c, hi, ig);
    }
}

// Face-intensity gradients, deterministic mode, last step: += into dL_dfaces_intense[B,F], poisoned like the other
// gradients of the call (det.cuh).  An intensity term beyond the range sets the shared overflow word, so it poisons
// those too.
__global__ void __launch_bounds__(256) tet_det_convert_intensity_kernel(size_t n, const uint32_t* __restrict__ gmax,
                                                                        TetIntGrad ig)
{
    griddep_wait();   // programmatic dependent launch: see dmr_launch (common.cuh)
    const size_t i = (size_t)blockIdx.x * 256 + threadIdx.x;
    if (i >= n) return;
    if (det_poisoned(gmax)) {
        ig.dL_dfint[i] = __int_as_float(0x7fc00000);
        return;
    }
    float sv, sg;
    det_scales(*gmax, sv, sg);
    if (sv == 0.0f) return;
    const long long* a = ig.det_fint + i;
    if (det_nonzero(a, ig.det_hi)) ig.dL_dfint[i] += (float)det_value(a, ig.det_hi, 1.0 / (double)sv);
}

// The march kernel of the intensity backward for the camera / vertex-position combination, with its stage.
static int tet_march_backward_intensity(const TetParams& p, cudaStream_t stream, dim3 grid, float* cam_rec,
                                        const TetVertGrad* vert, const TetIntGrad& ig, bool det)
{
    if (vert && cam_rec) {
        if (det) DMR_CUDA(dmr_launch(tet_march_bwd_cam_vert_int_det_kernel, grid, dim3(MARCH_THREADS), 0, stream, p, cam_rec, *vert, ig));
        else DMR_CUDA(dmr_launch(tet_march_bwd_cam_vert_int_kernel, grid, dim3(MARCH_THREADS), 0, stream, p, cam_rec, *vert, ig));
        DMR_LAUNCH_CHECK("tet_march_bwd_cam_vert_int_kernel");
    } else if (vert) {
        if (det) DMR_CUDA(dmr_launch(tet_march_bwd_vert_int_det_kernel, grid, dim3(MARCH_THREADS), 0, stream, p, *vert, ig));
        else DMR_CUDA(dmr_launch(tet_march_bwd_vert_int_kernel, grid, dim3(MARCH_THREADS), 0, stream, p, *vert, ig));
        DMR_LAUNCH_CHECK("tet_march_bwd_vert_int_kernel");
    } else if (cam_rec) {
        if (det) DMR_CUDA(dmr_launch(tet_march_bwd_cam_int_det_kernel, grid, dim3(MARCH_THREADS), 0, stream, p, cam_rec, ig));
        else DMR_CUDA(dmr_launch(tet_march_bwd_cam_int_kernel, grid, dim3(MARCH_THREADS), 0, stream, p, cam_rec, ig));
        DMR_LAUNCH_CHECK("tet_march_bwd_cam_int_kernel");
    } else {
        if (det) DMR_CUDA(dmr_launch(tet_march_bwd_int_det_kernel, grid, dim3(MARCH_THREADS), 0, stream, p, ig));
        else DMR_CUDA(dmr_launch(tet_march_bwd_int_kernel, grid, dim3(MARCH_THREADS), 0, stream, p, ig));
        DMR_LAUNCH_CHECK("tet_march_bwd_int_kernel");
    }
    return 0;
}

static int tet_int_stage(const float* cam_rec, const TetVertGrad* vert)
{
    return vert ? (cam_rec ? ST_TET_BWD_CAM_VERT_INT : ST_TET_BWD_VERT_INT) : (cam_rec ? ST_TET_BWD_CAM_INT : ST_TET_BWD_INT);
}

int tet_march_backward_deterministic(const TetParams& p, cudaStream_t stream, float* cam_rec, const TetVertGrad* vert,
                                     const TetIntGrad* fint, const float* dL_dalpha)
{
    dim3 grid((p.W + 7) / 8, (p.H + MARCH_ROWS - 1) / MARCH_ROWS, p.B);
    const size_t HW = (size_t)p.W * p.H;
    {
        ProfScope prof(dL_dalpha ? ST_TET_BWD_ALPHA
                       : fint    ? tet_int_stage(cam_rec, vert)
                       : vert    ? (cam_rec ? ST_TET_BWD_CAM_VERT : ST_TET_BWD_VERT) : (cam_rec ? ST_TET_BWD_CAM : ST_TET_BWD),
                       stream);
        count_launch(1);   // two kernels under one scope
        int rc = det_gmax(p.dL_dcolor, 3 * p.B * HW, p.dL_ddepth, p.B * HW, const_cast<uint32_t*>(p.det_gmax), stream);
        if (rc) return rc;
        if (dL_dalpha) {
            // the fixed-point scale covers max |dL_dalpha| too: a second maximum into the same word (order-independent)
            count_launch(1);
            if ((rc = det_gmax(dL_dalpha, p.B * HW, nullptr, 0, const_cast<uint32_t*>(p.det_gmax), stream))) return rc;
            DMR_CUDA(launch_tet_bwd_alpha<true>(p, stream, grid, cam_rec, vert, fint, dL_dalpha));
            DMR_LAUNCH_CHECK("tet_march_bwd_alpha_det_kernel");
        } else if (fint) {
            if ((rc = tet_march_backward_intensity(p, stream, grid, cam_rec, vert, *fint, true))) return rc;
        } else if (vert && cam_rec) {
            DMR_CUDA(dmr_launch(tet_march_bwd_cam_vert_det_kernel, dim3(grid), dim3(MARCH_THREADS), 0, stream, p, cam_rec, *vert));
            DMR_LAUNCH_CHECK("tet_march_bwd_cam_vert_det_kernel");
        } else if (vert) {
            DMR_CUDA(dmr_launch(tet_march_bwd_vert_det_kernel, dim3(grid), dim3(MARCH_THREADS), 0, stream, p, *vert));
            DMR_LAUNCH_CHECK("tet_march_bwd_vert_det_kernel");
        } else if (cam_rec) {
            DMR_CUDA(dmr_launch(tet_march_bwd_cam_det_kernel, dim3(grid), dim3(MARCH_THREADS), 0, stream, p, cam_rec));
            DMR_LAUNCH_CHECK("tet_march_bwd_cam_det_kernel");
        } else {
            DMR_CUDA(dmr_launch(tet_march_bwd_det_kernel, dim3(grid), dim3(MARCH_THREADS), 0, stream, p));
            DMR_LAUNCH_CHECK("tet_march_bwd_det_kernel");
        }
    }
    {
        ProfScope prof(ST_TET_BWD_FINISH, stream);
        DMR_CUDA(dmr_launch(tet_det_convert_kernel, dim3((unsigned)(((size_t)p.P + p.F + 255) / 256)), dim3(256), 0, stream, p));
        DMR_LAUNCH_CHECK("tet_det_convert_kernel");
    }
    if (vert) {
        ProfScope prof(ST_TET_VERT_FINISH, stream);
        DMR_CUDA(dmr_launch(tet_det_convert_position_kernel, dim3((p.P + 255) / 256), dim3(256), 0, stream, p.P, p.F,
                            p.det_gmax, *vert));
        DMR_LAUNCH_CHECK("tet_det_convert_position_kernel");
    }
    if (fint) {
        const size_t n = (size_t)p.B * p.F;
        ProfScope prof(ST_TET_INT_FINISH, stream);
        DMR_CUDA(dmr_launch(tet_det_convert_intensity_kernel, dim3((unsigned)((n + 255) / 256)), dim3(256), 0, stream, n,
                            p.det_gmax, *fint));
        DMR_LAUNCH_CHECK("tet_det_convert_intensity_kernel");
    }
    return 0;
}

int tet_march_backward(const TetParams& p, cudaStream_t stream, float* cam_rec, const TetVertGrad* vert,
                       const TetIntGrad* fint, const float* dL_dalpha)
{
    dim3 grid((p.W + 7) / 8, (p.H + MARCH_ROWS - 1) / MARCH_ROWS, p.B);
    if (dL_dalpha) {
        ProfScope prof(ST_TET_BWD_ALPHA, stream);
        DMR_CUDA(launch_tet_bwd_alpha<false>(p, stream, grid, cam_rec, vert, fint, dL_dalpha));
        DMR_LAUNCH_CHECK("tet_march_bwd_alpha_kernel");
    } else if (fint) {
        ProfScope prof(tet_int_stage(cam_rec, vert), stream);
        if (int rc = tet_march_backward_intensity(p, stream, grid, cam_rec, vert, *fint, false)) return rc;
    } else if (vert && cam_rec) {
        ProfScope prof(ST_TET_BWD_CAM_VERT, stream);
        DMR_CUDA(dmr_launch(tet_march_bwd_cam_vert_kernel, dim3(grid), dim3(MARCH_THREADS), 0, stream, p, cam_rec, *vert));
        DMR_LAUNCH_CHECK("tet_march_bwd_cam_vert_kernel");
    } else if (vert) {
        ProfScope prof(ST_TET_BWD_VERT, stream);
        DMR_CUDA(dmr_launch(tet_march_bwd_vert_kernel, dim3(grid), dim3(MARCH_THREADS), 0, stream, p, *vert));
        DMR_LAUNCH_CHECK("tet_march_bwd_vert_kernel");
    } else if (cam_rec) {
        ProfScope prof(ST_TET_BWD_CAM, stream);
        DMR_CUDA(dmr_launch(tet_march_bwd_cam_kernel, dim3(grid), dim3(MARCH_THREADS), 0, stream, p, cam_rec));
        DMR_LAUNCH_CHECK("tet_march_bwd_cam_kernel");
    } else {
        ProfScope prof(ST_TET_BWD, stream);
        DMR_CUDA(dmr_launch(tet_march_bwd_kernel, dim3(grid), dim3(MARCH_THREADS), 0, stream, p));
        DMR_LAUNCH_CHECK("tet_march_bwd_kernel");
    }
    {
        ProfScope prof(ST_TET_BWD_FINISH, stream);
        DMR_CUDA(dmr_launch(tet_grad_vertex_kernel, dim3((p.P + 255) / 256), dim3(256), 0, stream, p));
        DMR_LAUNCH_CHECK("tet_grad_vertex_kernel");
    }
    if (vert) {
        ProfScope prof(ST_TET_VERT_FINISH, stream);
        DMR_CUDA(dmr_launch(tet_grad_position_kernel, dim3((p.P + 255) / 256), dim3(256), 0, stream, p.P, *vert));
        DMR_LAUNCH_CHECK("tet_grad_position_kernel");
    }
    return 0;
}

int tet_camera_finish(const TetParams& p, const float* cam_rec, float* dL_dmv, float* dL_dproj, cudaStream_t stream)
{
    if (p.B <= 0) return 0;
    const int nrec = (int)tet_cam_records(1, p.W, p.H);
    ProfScope prof(ST_TET_CAM_FINISH, stream);
    DMR_CUDA(dmr_launch(tet_camera_finish_kernel, dim3(p.B), dim3(256), 0, stream, nrec, cam_rec, p.mv, p.proj, p.inv_mv,
                        p.inv_proj, dL_dmv, dL_dproj));
    DMR_LAUNCH_CHECK("tet_camera_finish_kernel");
    return 0;
}

}  // namespace dmr
