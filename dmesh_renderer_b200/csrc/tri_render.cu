// tri_render.cu -- per-tile compositing kernels of the tri renderer.
//
//   tri_render_fwd_kernel  replaces generateRaysCUDA + TRI_FORWARD::renderCUDA
//                          (cuda_rasterizer/forward.cu:184-231, 257-489)
//   tri_render_bwd_kernel  replaces TRI_BACKWARD::renderCUDA
//                          (cuda_rasterizer/backward.cu:9-421)
//
// One CTA per 16x16 tile, one thread per pixel; each warp owns an 8x4 pixel
// block.  Instances of the tile are staged in shared memory as 144-byte
// TriRecords (one contiguous copy per instance).
//
// Coverage, in both kernels: the thread that stages an instance decides once which of the tile's eight warp
// blocks it can touch (tile_block_mask: block bbox of the record + minimum of each edge function over a block,
// exact because the record is flagged overflow-free); every warp compacts its survivors in list order; ONE LANE
// PER SURVIVOR then evaluates the exact coverage of all 32 pixels of the block (block_coverage, the affine edge
// form documented at TriRecord, bit-identical to in_tri) and a 32x32 bit transpose across the warp turns the
// instance rows into one mask per pixel.  The shading arithmetic keeps the reference's expression order so that
// T, the early-termination decision and n_contrib are reproduced exactly.  Rays are recomputed per pixel (the
// reference stores 24 B/px and reads them back twice).
//
// Backward: see the design note above tri_render_bwd_kernel (sub-warp groups,
// sufficient statistics for the vertex-position gradient, transpose-reduction,
// one statistics record per (view, face) finished by tri_grad_finish_kernel)
// instead of the reference's 23 atomics per covered pixel.
#include "tri.cuh"
#include "det.cuh"

namespace dmr {

#define RB 256   // instances staged per round (one per thread)

// auxiliary.h:335-372
__device__ __forceinline__ void clamp_bary(float u, float v, float& uc, float& vc, int& code)
{
    if (u >= 0.0f && v >= 0.0f && u + v <= 1.0f) { uc = u; vc = v; code = 0; }
    else if (u <= 0.0f && v <= 0.0f) { uc = 0.0f; vc = 0.0f; code = 1; }
    else if ((u >= 1.0f && v <= 0.0f) || (v >= 0.0f && v <= u - 1.0f)) { uc = 1.0f; vc = 0.0f; code = 2; }
    else if ((u <= 0.0f && v >= 1.0f) || (u >= 0.0f && v >= u + 1.0f)) { uc = 0.0f; vc = 1.0f; code = 3; }
    else if (u <= 0.0f && v <= 1.0f && v >= 0.0f) { uc = 0.0f; vc = v; code = 4; }
    else if (u <= 1.0f && u >= 0.0f && v <= 0.0f) { uc = u; vc = 0.0f; code = 5; }
    else { uc = (1.0f + u - v) * 0.5f; vc = (1.0f - u + v) * 0.5f; code = 6; }
}

// Moeller-Trumbore (t,u,v), no inside test: auxiliary.h:255-286.
__device__ __forceinline__ bool ray_tri_tuv(float3 ro, float3 rd, float3 p0, float3 p1, float3 p2, float3& tuv,
                                            float& inv_denom_out)
{
    float3 T = ro - p0;
    float3 E1 = p1 - p0;
    float3 E2 = p2 - p0;
    float3 Pv = cross3(rd, E2);
    float3 Q = cross3(T, E1);
    float denom = dot3(Pv, E1);
    if (denom == 0.0f) return false;
    float inv_denom = 1.0f / denom;
    tuv.x = dot3(Q, E2) * inv_denom;
    tuv.y = dot3(Pv, T) * inv_denom;
    tuv.z = dot3(Q, rd) * inv_denom;
    inv_denom_out = inv_denom;
    return true;
}
__device__ __forceinline__ bool ray_tri_tuv(float3 ro, float3 rd, float3 p0, float3 p1, float3 p2, float3& tuv)
{
    float unused;
    return ray_tri_tuv(ro, rd, p0, p1, p2, tuv, unused);
}

// Which of the tile's eight 8x4 warp blocks (bit w <-> warp w: column w & 1, row w >> 1) can instance `e` touch?
// Evaluated ONCE per staged instance by the thread that stages it (the previous version let each of the 8 warps
// test every instance of the tile against its own block: 8 x 33 instructions per instance; this is ~80 for all
// eight).  Two conservative tests, both exact in the sense that they never drop a covered pixel:
//   * the block bbox of the record (DMR_REC_B*): blocks outside the triangle's pixel bounding box;
//   * the minimum of each edge function over a block (records flagged DMR_REC_SAFE only: no 32-bit overflow anywhere
//     on screen): a block where some edge function is non-negative everywhere.
__device__ __forceinline__ uint32_t tile_block_mask(const uint4 e0, const uint4 e1, const uint4 e2, int tx0, int ty0)
{
    const uint32_t fl = e0.w;
    // bbox: block columns tx0/8 + {0,1}, block rows ty0/4 + {0..3}
    const uint32_t nbx = (fl >> DMR_REC_NBX_SHIFT) & 15u, nby = (fl >> DMR_REC_NBY_SHIFT) & 15u;
    const uint32_t dx = (uint32_t)(tx0 >> 3) - ((fl >> DMR_REC_BX0_SHIFT) & 0x1ffu);
    const uint32_t dy = (uint32_t)(ty0 >> 2) - ((fl >> DMR_REC_BY0_SHIFT) & 0x3ffu);
    uint32_t xm = 3u, ym = 15u;
    if (nbx != DMR_REC_NB_UNBOUNDED) xm = (dx < nbx ? 1u : 0u) | (dx + 1u < nbx ? 2u : 0u);
    if (nby != DMR_REC_NB_UNBOUNDED)
        ym = (dy < nby ? 1u : 0u) | (dy + 1u < nby ? 2u : 0u) | (dy + 2u < nby ? 4u : 0u) | (dy + 3u < nby ? 8u : 0u);
    // bit j*2+i = xm bit i & ym bit j
    uint32_t mask = ((ym & 1u) ? xm : 0u) | ((ym & 2u) ? xm << 2 : 0u) | ((ym & 4u) ? xm << 4 : 0u) | ((ym & 8u) ? xm << 6 : 0u);
    if (!(fl & DMR_REC_SAFE) || mask == 0u) return mask;
    const int a[3] = { (int)e0.x, (int)e1.x, (int)e2.x }, bb[3] = { (int)e0.y, (int)e1.y, (int)e2.y };
    const int cc[3] = { (int)e0.z, (int)e1.z, (int)e2.z };
    int m[8] = { -1, -1, -1, -1, -1, -1, -1, -1 };
#pragma unroll
    for (int k = 0; k < 3; k++) {
        // minimum of edge k over block (i, j): at x = tx0 + 8i + (a < 0 ? 7 : 0), y = ty0 + 4j + (b < 0 ? 3 : 0)
        const int base = cc[k] + a[k] * (tx0 + (a[k] < 0 ? 7 : 0)) + bb[k] * (ty0 + (bb[k] < 0 ? 3 : 0));
        const int sx = 8 * a[k], sy = 4 * bb[k];
#pragma unroll
        for (int j = 0; j < 4; j++) { m[2 * j] &= base + j * sy; m[2 * j + 1] &= base + j * sy + sx; }
    }
    uint32_t em = 0;
#pragma unroll
    for (int w = 0; w < 8; w++) em |= m[w] < 0 ? (1u << w) : 0u;   // every edge can still be negative somewhere in the block
    return mask & em;
}

// Exact coverage of one instance over the warp's whole 8x4 pixel block, evaluated by ONE lane: bit p of the
// result <-> pixel (bx0 + (p & 7), by0 + (p >> 3)) is covered (in_tri true).  The three edge functions are
// stepped incrementally (ring operations mod 2^32, so the result is bit-identical to evaluating
// ea*x + eb*y + ec per pixel, overflow behaviour included); the pixels are visited from 31 down to 0 and
// every sign bit is shifted in with one funnel shift: 5 instructions per pixel.
__device__ __forceinline__ uint32_t block_coverage(const uint4 e0, const uint4 e1, const uint4 e2, int bx0, int by0)
{
    uint32_t r0 = e0.x * (uint32_t)(bx0 + 7) + e0.y * (uint32_t)(by0 + 3) + e0.z;
    uint32_t r1 = e1.x * (uint32_t)(bx0 + 7) + e1.y * (uint32_t)(by0 + 3) + e1.z;
    uint32_t r2 = e2.x * (uint32_t)(bx0 + 7) + e2.y * (uint32_t)(by0 + 3) + e2.z;
    uint32_t cov = 0;
#pragma unroll
    for (int y = 3; y >= 0; y--) {
        uint32_t s0 = r0, s1 = r1, s2 = r2;
#pragma unroll
        for (int x = 7; x >= 0; x--) {
            cov = __funnelshift_l(s0 & s1 & s2, cov, 1);   // (cov << 1) | sign(s0 & s1 & s2)
            if (x > 0) { s0 -= e0.x; s1 -= e1.x; s2 -= e2.x; }
        }
        if (y > 0) { r0 -= e0.y; r1 -= e1.y; r2 -= e2.y; }
    }
    return cov;
}

// 32x32 bit-matrix transpose across the lanes of a warp: lane i enters with row i (bit p = element (i, p)),
// lane p leaves with column p (bit i = element (i, p)).  Five butterfly steps; step j swaps the off-diagonal
// j x j blocks between lanes l and l ^ j.
__device__ __forceinline__ uint32_t transpose32(uint32_t x, int lane)
{
#pragma unroll
    for (int j = 16; j >= 1; j >>= 1) {
        const uint32_t m = j == 16 ? 0x0000ffffu : j == 8 ? 0x00ff00ffu : j == 4 ? 0x0f0f0f0fu : j == 2 ? 0x33333333u : 0x55555555u;
        const uint32_t y = __shfl_xor_sync(0xffffffffu, x, j);
        x = (lane & j) ? ((x & ~m) | ((y >> j) & m)) : ((x & m) | ((y << j) & ~m));
    }
    return x;
}


// Staging of a round: every warp copies the 32 records of ITS 32 instances (288 chunks of 16 B) cooperatively --
// chunk g = it * 32 + lane of the warp belongs to instance g / 9, whose face id comes from lane g / 9 by shuffle --
// so that nine consecutive lanes read one record's 144 contiguous bytes and a warp-wide LDG.128 touches ~7 cache
// lines.  The first version let thread t copy record t: every lane of a load instruction hit a different line,
// 32 L1 wavefronts per instruction, and ncu showed the L1 data pipe (l1tex__data_pipe_lsu_wavefronts), not the
// issue slots, as the busiest unit of both render kernels (70 % / 67 % of peak at C4, a quarter of it this
// gather).  `nvw` = instances of the round that fall to this warp (<= 0: none), `face` = this lane's face id.
__device__ __forceinline__ void stage_records_warp(uint4* __restrict__ dstw, const TriRecord* __restrict__ recs, uint32_t face,
                                                   int nvw, int lane)
{
    // asynchronous copies (cp.async, SASS LDGSTS): global -> shared without a round trip through 36 registers
    const uint32_t dst0 = (uint32_t)__cvta_generic_to_shared(dstw);
#pragma unroll
    for (int it = 0; it < 9; it++) {
        const unsigned g = it * 32 + lane, rr = g / 9u, part = g - rr * 9u;
        const uint32_t fr = __shfl_sync(0xffffffffu, face, rr);
        if ((int)rr < nvw)
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" :: "r"(dst0 + g * 16u),
                         "l"(reinterpret_cast<const uint4*>(recs + fr) + part) : "memory");
    }
    asm volatile("cp.async.commit_group;\n\tcp.async.wait_group 0;" ::: "memory");
    __syncwarp();
}

constexpr int HB = 256;          // staged instances a warp compacts / rasterises / shades in one go (measured: 128 -> 256 = -5 % at C4, -3 % at C2, +-0 at C5)
constexpr int HS = HB / 32;      // 32-entry slices of the compacted list of such a pass

// (Measured and rejected, round 2: L2 prefetch -- prefetch.global.L2, SASS CCTL.E.PF2, one per 32-byte sector -- of the
// record each thread stages in the NEXT round and of the first round of the tile two waves of CTAs later in the grid.
// ncu had 24 % of the forward kernel's warp samples at the staging loads and the barrier behind them (a dependent
// chain range -> face id -> scattered 144-byte gather that misses L2 half of the time), but the prefetches cost more
// than the latency they hide: C4 forward 1833 -> 1903 us, backward 3602 -> 3766 us; C5 forward 443 -> 822 us.  The
// bulk form cp.async.bulk.prefetch.L2 is a uniform-datapath instruction -- per-lane addresses compile to a
// 32-iteration loop around it.  Also rejected: fetching the face id of the instance a thread stages in the NEXT round
// one round ahead (one register; staging becomes a single dependent gather): C4 forward 1831 -> 1889 us.  The
// staging latency is already covered by the other three CTAs of the SM.  And: eight ballots in the staging warp that
// hand every warp block its "which of these 32 staged instances can touch me" word, so that a compaction step is a
// broadcast load and a bit test instead of a byte load, shift, test and vote: C4 forward 1578 -> 1620 us.)

// (Measured and rejected, round 2: per-(view, face) constants of the ray-triangle system -- E2 x E1, E2 x T, T x E1 formed
// once per staged instance, so that a covered pixel needs three dot products instead of Moeller-Trumbore's two cross
// products and four dots.  -4 % forward, -3 % backward at C4, but it is the same real number with DIFFERENT roundings:
// for triangles seen edge-on (det tiny against |E1||E2|) the reference's own (u, v) carry a large relative error, and
// only the reference's exact operation order reproduces it.  C1, C2 and C4 stayed within 1e-5; C5 (4 M triangles,
// thousands of slivers per image) differed by up to 7e-4 in colour.  Parity wins: ray_tri_tuv stays.
// Second attempt, also rejected: hoisting only the pixel-independent HALF of ray_tri_tuv (T = ro - p0, E1, E2, T x E1
// are per (view, face)) into the staging code, same operations on the same operands.  The compiler fuses a*b - c*d
// either way round depending on context, so the hoisted cross product first differed from the reference by an ulp
// (C5 failed again); with every dot / cross pinned to explicit fma forms parity held at all configs -- but the 15
// instructions saved per hit bought nothing: forward 1840 -> 1886 us, backward 3677 -> 3689 us at C4.)

// Forward.  Per round of RB staged instances every warp works through its 8x4 pixel block in passes of HB
// instances:
//   (1) cull + compact: one lane per instance tests the instance against the whole block (minimum of each edge
//       function over the block, exact for overflow-free records); the survivors' positions are compacted, in list
//       order, into a per-warp index list -- a tile's list holds every face that touches the 16x16 tile, only
//       ~1/3 of them reach a given 8x4 block;
//   (2) rasterise: one lane per SURVIVOR evaluates the exact coverage of all 32 pixels (block_coverage, 5
//       instructions per pixel) and a 32x32 bit transpose turns the 32 instance rows into one mask per pixel.
//       (The previous version let all 32 lanes test their own pixel against one survivor at a time: 25 warp
//       instructions per survivor and 28 % of the kernel at C2; this is ~7 per survivor.)
//   (3) shade: every lane pops ITS next covered instance from its masks, so the lanes of a warp shade different
//       faces in the same SIMD pass and per pixel the list order (front to back) is unchanged.  The masks of a
//       whole pass are known up front, so a lane with few hits in one 32-instance slice moves straight on to the
//       next one: the number of SIMD passes is the largest per-pixel hit count over HB instances, not the sum of
//       the per-slice maxima (the shading path ran at 15 of 32 lanes before).
constexpr int DMR_TRI_FWD_MINB = 4;
__global__ void __launch_bounds__(256, DMR_TRI_FWD_MINB) tri_render_fwd_kernel(TriRenderParams p)
{
    griddep_wait();   // programmatic dependent launch: see dmr_launch (common.cuh)
    __shared__ uint4 s_rec[RB * 9];
    __shared__ unsigned char s_bmask[RB];         // [staged instance]: warp blocks of the tile it can touch (tile_block_mask)
    __shared__ unsigned char s_cidx[8 * HB];      // [warp][compacted position] -> position in the staged round
    __shared__ uint32_t s_pmask[8 * HS * 32];     // [warp][slice][lane]: covered compacted instances of the lane's pixel
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int b = blockIdx.z;
    const int tiles_x = gridDim.x, tiles_y = gridDim.y;
    const int bx0 = blockIdx.x * DMR_TILE + (warp & 1) * 8, by0 = blockIdx.y * DMR_TILE + (warp >> 1) * 4;
    const uint32_t px = bx0 + (lane & 7);
    const uint32_t py = by0 + (lane >> 3);
    const bool inside = px < (uint32_t)p.W && py < (uint32_t)p.H;
    bool done = !inside;
    const uint32_t lt_mask = (1u << lane) - 1u;
    unsigned char* const cidx = s_cidx + warp * HB;
    uint32_t* const pmask = s_pmask + warp * HS * 32;

    float3 ro, rd;
    pixel_ray<false>(p.inv_mv + 16 * b, p.inv_proj + 16 * b, px + 0.5f, py + 0.5f, p.W, p.H, ro, rd);

    const uint2 range = p.ranges[(size_t)b * tiles_x * tiles_y + blockIdx.y * tiles_x + blockIdx.x];
    const int total = (int)(range.y - range.x);
    const int rounds = (total + RB - 1) / RB;

    float T = 1.0f, pT = 1.0f;
    uint32_t last_contributor = 0;
    float C0 = 0, C1 = 0, C2 = 0, D = 0;

    for (int r = 0; r < rounds; r++) {
        if (__syncthreads_count(done) == 256) break;
        {   // stage (stage_records_warp), then thread t finds the warp blocks of the tile that instance t can touch
            const int nvw = min(32, total - r * RB - warp * 32);
            uint32_t face = 0u;
            if (lane < nvw) face = p.face_list[range.x + (uint32_t)r * RB + tid];
            stage_records_warp(s_rec + warp * 32 * 9, p.records + (size_t)b * p.F, face, nvw, lane);
            uint32_t bm = 0;
            if (lane < nvw)
                bm = tile_block_mask(s_rec[tid * 9 + 0], s_rec[tid * 9 + 1], s_rec[tid * 9 + 2], blockIdx.x * DMR_TILE, blockIdx.y * DMR_TILE);
            s_bmask[tid] = (unsigned char)bm;
        }
        __syncthreads();
        const int cnt = min(RB, total - r * RB);
        for (int h0 = 0; h0 < cnt; h0 += HB) {
            if (__all_sync(0xffffffffu, done)) break;
            const int hcnt = min(HB, cnt - h0);
            // (1) compact the instances whose block mask has this warp's bit (unstaged slots carry mask 0)
            int ncomp = 0;
            for (int c0 = 0; c0 < hcnt; c0 += 32) {
                const int jl = h0 + c0 + lane;
                const bool keep = (s_bmask[jl] >> warp) & 1u;
                const unsigned m = __ballot_sync(0xffffffffu, keep);
                if (keep) cidx[ncomp + __popc(m & lt_mask)] = (unsigned char)jl;
                ncomp += __popc(m);
            }
            __syncwarp();
            const int nsl = (ncomp + 31) >> 5;
            // (2) rasterise the survivors, one lane per instance, and transpose to one mask per pixel
            for (int sl = 0; sl < nsl; sl++) {
                const int jc = (sl << 5) + lane;
                uint32_t cov = 0;
                if (jc < ncomp) {
                    const int jl = cidx[jc];
                    cov = block_coverage(s_rec[jl * 9 + 0], s_rec[jl * 9 + 1], s_rec[jl * 9 + 2], bx0, by0);
                }
                const uint32_t col = transpose32(cov, lane);
                pmask[(sl << 5) + lane] = done ? 0u : col;      // read back by this lane only
            }
            // (3) shade
            int sl = 0;
            uint32_t mine = nsl > 0 ? pmask[lane] : 0u;
            for (;;) {
                while (mine == 0u && sl + 1 < nsl) { sl++; mine = pmask[(sl << 5) + lane]; }
                if (!__any_sync(0xffffffffu, mine != 0u)) break;
                if (mine != 0u) {
                    const int bit = __ffs(mine) - 1;
                    mine &= mine - 1;
                    const int j = cidx[(sl << 5) + bit];
                    const float4* sh = reinterpret_cast<const float4*>(s_rec + j * 9 + 3);   // the six shading chunks
                    const float4 a0 = sh[0], a1 = sh[1], a2 = sh[2];                         // (v_k, opacity | intensity | -)
                    float3 tuv = f3(0, 0, 0);
                    const bool hit = ray_tri_tuv(ro, rd, f3(a0.x, a0.y, a0.z), f3(a1.x, a1.y, a1.z), f3(a2.x, a2.y, a2.z), tuv);
                    if (hit) {
                        float uc, vc;
                        int code;
                        clamp_bary(tuv.y, tuv.z, uc, vc, code);
                        float i0 = 1 - uc - vc, i1 = uc, i2 = vc;
                        const float4 k0 = sh[3], k1 = sh[4], k2 = sh[5];                     // (colour_k, depth_k)
                        const float intense = a1.w;
                        // forward.cu:442-451
                        float c0_ = i0 * k0.x + i1 * k1.x + i2 * k2.x; c0_ = c0_ * intense;
                        float c1_ = i0 * k0.y + i1 * k1.y + i2 * k2.y; c1_ = c1_ * intense;
                        float c2_ = i0 * k0.z + i1 * k1.z + i2 * k2.z; c2_ = c2_ * intense;
                        float iD = i0 * k0.w + i1 * k1.w + i2 * k2.w;
                        const float alpha = a0.w;
                        float test_T = T * (1 - alpha);
                        C0 += c0_ * alpha * T;
                        C1 += c1_ * alpha * T;
                        C2 += c2_ * alpha * T;
                        D += iD * alpha * T;
                        pT = T;
                        T = test_T;
                        last_contributor = (uint32_t)(r * RB + j + 1);
                        if (T < DMR_T_EPS) { done = true; mine = 0u; sl = nsl; }
                    }
                }
            }
            __syncwarp();   // the next pass overwrites the index list
        }
    }

    if (inside) {
        const size_t HW = (size_t)p.W * p.H;
        const size_t pix = (size_t)py * p.W + px;
        const size_t bpix = (size_t)b * HW + pix;
        p.prev_T[bpix] = pT;
        p.final_T[bpix] = T;
        p.n_contrib[bpix] = last_contributor;
        p.out_color[(size_t)b * 3 * HW + 0 * HW + pix] = C0 + T * p.bg[0];
        p.out_color[(size_t)b * 3 * HW + 1 * HW + pix] = C1 + T * p.bg[1];
        p.out_color[(size_t)b * 3 * HW + 2 * HW + pix] = C2 + T * p.bg[2];
        p.out_depth[bpix] = D + T * 1.0f;
    }
}

// ---------------------------------------------------------------------------
// backward
// ---------------------------------------------------------------------------

// 32-bit shared-memory load the compiler cannot merge into a neighbouring vector load
__device__ __forceinline__ float lds_f32(const float* p)
{
    float v;
    asm("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"((uint32_t)__cvta_generic_to_shared(p)));
    return v;
}

// auxiliary.h:374-400
__device__ __forceinline__ void clamp_bary_grad(int code, float& duc_du, float& duc_dv, float& dvc_du, float& dvc_dv)
{
    dvc_du = 0.0f; duc_dv = 0.0f;
    if (code == 0) { duc_du = 1.0f; dvc_dv = 1.0f; }
    else if (code == 1 || code == 2 || code == 3) { duc_du = 0.0f; dvc_dv = 0.0f; }
    else if (code == 4) { duc_du = 0.0f; dvc_dv = 1.0f; }
    else if (code == 5) { duc_du = 1.0f; dvc_dv = 0.0f; }
    else { duc_du = 0.5f; dvc_du = -0.5f; duc_dv = -0.5f; dvc_dv = 0.5f; }
}

// One step of the transpose-reduction: lanes whose bit `M` is clear keep the lower
// N values and send the upper N, the others the opposite; afterwards v[0..N) holds
// the pairwise sums.
template <int N, int M>
__device__ __forceinline__ void xreduce_step(float* v, bool hi)
{
#pragma unroll
    for (int k = 0; k < N; k++) {
        float send = hi ? v[k] : v[k + N];
        float keep = hi ? v[k + N] : v[k];
        v[k] = keep + __shfl_xor_sync(0xffffffffu, send, M);
    }
}

// Position of logical statistic i (0..23) inside the 24-float record.  The transpose-reduction leaves lane class
// c = lane & 1 of a group with the twelve sums 12c .. 12c + 11, which it adds as three 16-byte vector reductions.
// Reduction k of class c goes to bytes 32k + 16c: the two lanes of a group fill ONE 32-byte sector per instruction,
// three sector operations per group and pass at the L2 (round 1's layout -- quads 2c, 2c + 1 and the pair 2c, 2c + 1 of
// the last 32 bytes -- cost five, a class-major layout six: C5, whose 4 M statistics records do not stay in L2, ran
// its backward kernel 12 % slower with the latter), and the three addresses of a lane are one base + immediates.
__host__ __device__ constexpr int stat_slot(int i) { return 8 * ((i % 12) / 4) + 4 * (i / 12) + (i % 4); }
constexpr bool stat_slot_is_permutation()
{
    unsigned seen = 0;
    for (int i = 0; i < 24; i++) seen |= 1u << stat_slot(i);
    return seen == 0xffffffu;
}
static_assert(stat_slot_is_permutation(), "stat_slot must map the 24 statistics onto the 24 floats of a record");

// Backward design
// ---------------
// * A warp owns an 8x4 pixel block (pixel of lane p: x = p & 7, y = p >> 3), split into 16 GROUPS of 2
//   horizontally adjacent pixels.  Cull, compaction and exact per-pixel coverage masks are built exactly as in
//   the forward kernel (one lane per surviving instance + 32x32 bit transpose); a group's candidate list is the
//   OR of its two pixel masks, so finding a group's next instance is one count-leading-zeros -- no edge
//   functions and no votes inside the walk (the previous version popped candidates of a conservative 2x1
//   sub-block cull and re-tested them per pixel: 20 % of the kernel's instructions at C2, plus 8 % for the cull).
//   Each group walks ITS OWN list, back to front, so the groups shade different faces in the same SIMD pass.
// * Vertex-position gradients are not formed per pixel.  With u = A/D, A = rd.(E2xT), D = rd.(E2xE1) and
//   the reference's "v" derivative (ray_tri_intersection_grad, auxiliary.h:288-333, actually the derivative
//   of t = Nt/D, Nt = (TxE1).E2), the per-face sums only need
//       S1  = sum dL_du/D * rd          S24 = sum (dL_du*u + dL_dv*t)/D * rd          S3 = sum dL_dv/D
//   (7 floats); tri_grad_finish_kernel turns them into dL_dp0..2 once per (view, face):
//       g_E1 = S3 (E2xT) - S24xE2,  g_E2 = TxS1 - E1xS24 + S3 (TxE1),  g_T = S1xE2 + S3 (E1xE2).
//   This is the same derivative the reference evaluates per covered pixel with ~150 instructions.
// * All 21 per-hit terms of a group are reduced over its two lanes with a transpose-reduction (12 shuffles)
//   and added to ONE contiguous 96-byte statistics record per (view, face) with vector reductions (red.v4)
//   instead of 21 scalar reductions per lane.
// Statistics (logical order, 24 floats; memory position = stat_slot(i)):
//   S1[3] S24[3] S3 dL_dopacity dL_dintense dL_ddepth[3] dL_dcolor[3][3] pad[3]
// History of the group size, measured on B200 with the earlier find loop (us, C2 / C5 / C4 with 8 views):
// 8 lanes 537 / 1172 / 7808, 4 lanes 476 / 1079 / 6752, 2 lanes 459 / 1057 / 6532.  One lane per group would need
// no shuffles at all but 6 vector reductions per covered pixel, which the LSU/L2 cannot sustain
// (tools/ubench_red.cu).
// Resident CTAs per SM.  3 (80 registers, no spills) against 4 (64 registers, 80 bytes of spill): the kernel issues
// on only ~64 % of the cycles with 5.6 warps per scheduler and its stalls spread evenly over memory, barrier and
// dependency waits, so two more warps per scheduler win slightly -- C4 3677 -> 3640 us, C5 788 -> 766 us, C2 291 -> 289 us.
constexpr int DMR_TRI_BWD_MINB = 4;
// Camera gradients (CAM = true; DESIGN.md 3.3).  The rays are the only place the camera enters a pixel's colour and
// depth: ro = inv_mv[12..14], rd = d / (|d| + 1e-7), d = L pv, pv = (inv_proj (nx, ny, -1, 1)).xyz, L = the linear
// part of inv_mv.  Per covered hit, with T = ro - p0, E1, E2, P = rd x E2, Q = T x E1, D = P.E1, u = P.T / D and
// v = Q.rd / D, each lane (one pixel) accumulates
//     g_ro += (dL_du P + dL_dv (E1 x rd)) / D
//     g_rd += (dL_du (E2 x T) + dL_dv Q - (dL_du u + dL_dv v) (E2 x E1)) / D
// -- the exact derivative of v, not the reference's t-derivative the vertex-position statistics keep.  After the walk
// the lane chains its pixel into the 24 nonzero partials of dL/dinv_mv and dL/dinv_proj (cam_record_slot), the CTA
// sums them in a fixed order and stores ONE 96-byte record per (view, tile): no float atomics, so the camera
// gradients are reproducible in both modes.  tri_camera_finish_kernel sums a view's records and applies the inverse.
#define DMR_CAM_REC 24
// Exact vertex-position gradients (EXACT = true, opt-in; DESIGN.md 3.3).  The statistics differentiate the v the
// forward pass uses instead of the reference's t: S24 takes dL_dv * v in place of dL_dv * t, and S3 becomes the
// vector S3v = sum dL_dv / D * rd, whose y and z go to the pad slots 21 and 22 of the record (logical 6 keeps x).
// Record size, reduction and stores are unchanged; tri_grad_finish_body<.., EXACT> applies the matching formula.
// Alpha cotangent (ALPHA = true, opt-in; DESIGN.md 3.3).  alpha = 1 - T_final, and T_final is the factor the forward
// pass multiplies the background by, so dL/dalpha enters exactly where the background term does: the per-pixel
// constant bg . dL_dC + dL_dD becomes bg . dL_dC + dL_dD - dL_dalpha.  One more load per pixel, before the walk.
// The cotangent arrives as a parameter pack, empty for every other instantiation: those keep exactly their two
// parameters (an unused defaulted pointer changed ptxas's register assignment in the camera kernels).
template <bool DET, bool CAM, bool EXACT = false, bool ALPHA = false, class... AlphaPtr>
__device__ __forceinline__ void tri_render_bwd_body(const TriRenderParams& p, float* __restrict__ cam_tiles,
                                                    AlphaPtr... dL_dalpha)
{
    __shared__ uint4 s_rec[RB * 9];      // staged records; two vertex-id slots (unused here: tri_grad_finish_kernel reads the
                                         // global record) carry the face id and 1 / (1 - opacity) of the instance
    __shared__ int s_max[8];
    __shared__ unsigned char s_bmask[RB];         // [staged instance]: warp blocks of the tile it can touch (tile_block_mask)
    __shared__ unsigned char s_cidx[8 * HB];      // [warp][compacted position] -> position in the chunk
    __shared__ uint32_t s_pmask[8 * HS * 32];     // [warp][slice][lane]: covered compacted instances of the lane's pixel
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int b = blockIdx.z;
    const int tiles_x = gridDim.x, tiles_y = gridDim.y;
    const int bx0 = blockIdx.x * DMR_TILE + (warp & 1) * 8, by0 = blockIdx.y * DMR_TILE + (warp >> 1) * 4;
    const uint32_t px = bx0 + (lane & 7);
    const uint32_t py = by0 + (lane >> 3);
    const bool inside = px < (uint32_t)p.W && py < (uint32_t)p.H;
    const size_t HW = (size_t)p.W * p.H;
    const size_t pix = (size_t)py * p.W + px;
    const size_t bpix = (size_t)b * HW + pix;
    const uint32_t lt_mask = (1u << lane) - 1u;
    unsigned char* const cidx = s_cidx + warp * HB;
    uint32_t* const pmask = s_pmask + warp * HS * 32;

    float3 ro, rd;
    pixel_ray<false>(p.inv_mv + 16 * b, p.inv_proj + 16 * b, px + 0.5f, py + 0.5f, p.W, p.H, ro, rd);

    const uint2 range = p.ranges[(size_t)b * tiles_x * tiles_y + blockIdx.y * tiles_x + blockIdx.x];

    const float T_final = inside ? p.final_T[bpix] : 0;
    const float prev_T_final = inside ? p.prev_T[bpix] : 0;
    const int last_contributor = inside ? (int)p.n_contrib[bpix] : 0;
    float T = prev_T_final;
    bool T_first = true;

    float dLc0 = 0, dLc1 = 0, dLc2 = 0, dLd = 0;
    if (inside) {
        dLc0 = p.dL_dcolor[(size_t)b * 3 * HW + 0 * HW + pix];
        dLc1 = p.dL_dcolor[(size_t)b * 3 * HW + 1 * HW + pix];
        dLc2 = p.dL_dcolor[(size_t)b * 3 * HW + 2 * HW + pix];
        dLd = p.dL_ddepth[bpix];
    }
    const float bg0 = p.bg[0], bg1 = p.bg[1], bg2 = p.bg[2];
    // backward.cu:293-298
    float bg_dot = 0; bg_dot += bg0 * dLc0; bg_dot += bg1 * dLc1; bg_dot += bg2 * dLc2;
    float bd_dot = 0; bd_dot += 1.0 * dLd;
    if constexpr (ALPHA) {
        static_assert(sizeof...(AlphaPtr) == 1, "ALPHA takes the cotangent pointer");
        const float* const dla = (dL_dalpha, ...);
        if (inside) bd_dot -= dla[bpix];
    }
    const float bgk = -T_final * (bg_dot + bd_dot), bgk1 = -prev_T_final * (bg_dot + bd_dot);

    float acc0 = 0, acc1 = 0, acc2 = 0, accd = 0;
    float last_alpha = 0, lc0 = 0, lc1 = 0, lc2 = 0, ld = 0;
    float3 g_ro = f3(0, 0, 0), g_rd = f3(0, 0, 0);   // CAM only: dL/dro, dL/drd of this pixel

    // The tile walks only the prefix some pixel of it composited; a warp only its own.
    int warp_last = last_contributor;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) warp_last = max(warp_last, __shfl_xor_sync(0xffffffffu, warp_last, o));
    if (lane == 0) s_max[warp] = warp_last;
    __syncthreads();
    int tile_last = 0;
#pragma unroll
    for (int w = 0; w < 8; w++) tile_last = max(tile_last, s_max[w]);
    const int nchunk = (tile_last + RB - 1) / RB;   // chunk c covers list positions [c*RB, c*RB+RB)

    const bool h1 = lane & 1;
    float* const stats = p.grad_stats;
    float det_sv = 0.0f, det_sg = 0.0f;
    if (DET) det_scales(*p.det_gmax, det_sv, det_sg);

    for (int c = nchunk - 1; c >= 0; c--) {
        __syncthreads();
        {   // stage (stage_records_warp); the owner of an instance then adds the face id and 1 / (1 - alpha) to the
            // staged copy and finds the warp blocks of the tile the instance can touch
            const int nvw = min(32, tile_last - c * RB - warp * 32);
            uint32_t face = 0u;
            if (lane < nvw) face = p.face_list[range.x + c * RB + tid];
            stage_records_warp(s_rec + warp * 32 * 9, p.records + (size_t)b * p.F, face, nvw, lane);
            uint32_t bm = 0;
            if (lane < nvw) {
                uint32_t* rw = reinterpret_cast<uint32_t*>(s_rec + tid * 9);
                rw[7] = (uint32_t)b * (uint32_t)p.F + face;                                     // q1.w: i0 -> index of the (view, face) statistics record
                rw[23] = __float_as_uint(1.0f / (1.0f - __uint_as_float(rw[15])));             // q5.w: i2 -> 1 / (1 - opacity)
                bm = tile_block_mask(s_rec[tid * 9 + 0], s_rec[tid * 9 + 1], s_rec[tid * 9 + 2], blockIdx.x * DMR_TILE, blockIdx.y * DMR_TILE);
            }
            s_bmask[tid] = (unsigned char)bm;
        }
        __syncthreads();
        const int cnt = min(RB, warp_last - c * RB);       // this warp's share of the chunk
        // reference: skip when contributor >= last_contributor (backward.cu:192-194); in chunk-relative positions
        const int limit = last_contributor - c * RB;

        for (int h0 = cnt > 0 ? ((cnt - 1) / HB) * HB : -1; h0 >= 0; h0 -= HB) {
            const int hcnt = min(HB, cnt - h0);
            // (1) compact, in list order, the instances whose block mask has this warp's bit
            int ncomp = 0;
            for (int c0 = 0; c0 < hcnt; c0 += 32) {
                const int jl = h0 + c0 + lane;
                const bool keep = c0 + lane < hcnt && ((s_bmask[jl] >> warp) & 1u);
                const unsigned m = __ballot_sync(0xffffffffu, keep);
                if (keep) cidx[ncomp + __popc(m & lt_mask)] = (unsigned char)jl;
                ncomp += __popc(m);
            }
            __syncwarp();
            const int nsl = (ncomp + 31) >> 5;
            // (2) exact coverage masks per pixel; instances at or behind the pixel's last contributor are dropped
            for (int sl = 0; sl < nsl; sl++) {
                const int jc = (sl << 5) + lane;
                uint32_t cov = 0;
                if (jc < ncomp) {
                    const int jl = cidx[jc];
                    cov = block_coverage(s_rec[jl * 9 + 0], s_rec[jl * 9 + 1], s_rec[jl * 9 + 2], bx0, by0);
                }
                uint32_t col = transpose32(cov, lane);
                if (col != 0u) {
                    const int n_here = min(32, ncomp - (sl << 5));
                    if ((int)cidx[(sl << 5) + n_here - 1] >= limit) {
                        int lo = 0, hi = n_here;           // first entry of the slice at or behind the limit
                        while (lo < hi) {
                            const int mid = (lo + hi) >> 1;
                            if ((int)cidx[(sl << 5) + mid] < limit) lo = mid + 1; else hi = mid;
                        }
                        if (lo < 32) col &= (1u << lo) - 1u;
                    }
                }
                pmask[(sl << 5) + lane] = col;
            }
            __syncwarp();

            // (3) walk, back to front: both lanes of a group hold the group's candidate mask `gm` and its own
            //     pixel's mask `mine` of the slice the group is working on
            int sl = nsl;
            uint32_t mine = 0u, gm = 0u;
            for (;;) {
                while (gm == 0u && sl > 0) {
                    sl--;
                    mine = pmask[(sl << 5) + lane];
                    gm = mine | pmask[(sl << 5) + (lane ^ 1)];
                }
                const bool have = gm != 0u;
                if (!__any_sync(0xffffffffu, have)) break;
                bool cov = false;
                int j = 0;
                if (have) {
                    const int bit = 31 - __clz(gm);
                    gm &= ~(1u << bit);
                    cov = (mine >> bit) & 1u;
                    j = cidx[(sl << 5) + bit];
                }

                // ---- shade: lanes with a covered pixel evaluate the gradient terms of their group's face
                float v[24];
#pragma unroll
                for (int k = 0; k < 24; k++) v[k] = 0.0f;
                if (cov) {
                    const float4* sh = reinterpret_cast<const float4*>(s_rec + j * 9 + 3);   // the six shading chunks
                    const float4 a0 = sh[0], a1 = sh[1], a2 = sh[2];                         // (v_k, opacity | intensity | 1 / (1 - opacity))
                    float3 tuv = f3(0, 0, 0);
                    float inv_denom = 0.0f;
                    const bool hit = ray_tri_tuv(ro, rd, f3(a0.x, a0.y, a0.z), f3(a1.x, a1.y, a1.z), f3(a2.x, a2.y, a2.z), tuv, inv_denom);
                    if (hit) {
                        float uc, vc;
                        int code;
                        clamp_bary(tuv.y, tuv.z, uc, vc, code);
                        const float i0 = 1 - uc - vc, i1 = uc, i2 = vc;
                        const float4 q6 = sh[3], q7 = sh[4], q8 = sh[5];                     // (colour_k, depth_k)
                        // (scalar loads on purpose: taking these three from the .w lanes of a0..a2 keeps them live across the
                        // hit test and costs the 64-register kernel three spill accesses per pass: C4 3316 -> 3408 us;
                        // re-measured after the statistics addressing freed registers -- one extra spill load per pass
                        // instead of three: C4 3133 -> 3173 us, C5 699 -> 707 us)
                        const float intense = lds_f32(&sh[1].w);
                        const float alpha = lds_f32(&sh[0].w);
                        const float raw0 = i0 * q6.x + i1 * q7.x + i2 * q8.x;
                        const float raw1 = i0 * q6.y + i1 * q7.y + i2 * q8.y;
                        const float raw2 = i0 * q6.z + i1 * q7.z + i2 * q8.z;
                        const float iC0 = raw0 * intense, iC1 = raw1 * intense, iC2 = raw2 * intense;
                        const float iD = i0 * q6.w + i1 * q7.w + i2 * q8.w;

                        // backward.cu:244-252.  1/(1-alpha) is formed once per staged instance and multiplied, instead
                        // of the reference's two divisions per covered pixel (here and in the background term,
                        // backward.cu:299-308); T and the background term change by an ulp per step.
                        const float rcpa = lds_f32(&sh[2].w);
                        if (!T_first) T = T * rcpa;
                        T_first = false;

                        float dL_dalpha = 0.0f;
                        // colour, backward.cu:262-272
                        acc0 = last_alpha * lc0 + (1.f - last_alpha) * acc0; lc0 = iC0;
                        const float dic0 = dLc0 * alpha * T; dL_dalpha += (iC0 - acc0) * dLc0;
                        acc1 = last_alpha * lc1 + (1.f - last_alpha) * acc1; lc1 = iC1;
                        const float dic1 = dLc1 * alpha * T; dL_dalpha += (iC1 - acc1) * dLc1;
                        acc2 = last_alpha * lc2 + (1.f - last_alpha) * acc2; lc2 = iC2;
                        const float dic2 = dLc2 * alpha * T; dL_dalpha += (iC2 - acc2) * dLc2;
                        // depth, backward.cu:275-284
                        accd = last_alpha * ld + (1.f - last_alpha) * accd; ld = iD;
                        const float did = dLd * alpha * T; dL_dalpha += (iD - accd) * dLd;

                        dL_dalpha *= T;
                        last_alpha = alpha;
                        // background term, backward.cu:299-308: (-T_final / (1 - alpha)) * (bg . dL_dC) and the same factor
                        // times dL_dD.  The pixel constants -T_final * (bg . dL_dC + dL_dD) and its alpha == 1 counterpart
                        // are formed once (two live registers instead of four; one rounding apart from the reference's
                        // two separate products, far inside the gradient tolerance)
                        dL_dalpha += (alpha == 1.0f) ? bgk1 : bgk * rcpa;

                        // backward.cu:327-349.  The per-term products are the reference's; the common factor
                        // dic*intense is formed once (the reference multiplies (x*dic)*intense per term: one
                        // rounding apart, far inside the 1e-4 gradient tolerance).
                        const float dI0 = dic0 * intense, dI1 = dic1 * intense, dI2 = dic2 * intense;
                        const float dL_di0 = q6.x * dI0 + q6.y * dI1 + q6.z * dI2 + q6.w * did;
                        const float dL_di1 = q7.x * dI0 + q7.y * dI1 + q7.z * dI2 + q7.w * did;
                        const float dL_di2 = q8.x * dI0 + q8.y * dI1 + q8.z * dI2 + q8.w * did;
                        v[12] = i0 * dI0; v[13] = i0 * dI1; v[14] = i0 * dI2;
                        v[15] = i1 * dI0; v[16] = i1 * dI1; v[17] = i1 * dI2;
                        v[18] = i2 * dI0; v[19] = i2 * dI1; v[20] = i2 * dI2;
                        v[9] = i0 * did; v[10] = i1 * did; v[11] = i2 * did;
                        v[7] = dL_dalpha;
                        v[8] = raw0 * dic0 + raw1 * dic1 + raw2 * dic2;

                        // backward.cu:354-369: chain through the clamp
                        float duc_du, duc_dv, dvc_du, dvc_dv;
                        clamp_bary_grad(code, duc_du, duc_dv, dvc_du, dvc_dv);
                        // i0 = 1 - uc - vc, i1 = uc, i2 = vc: dL/duc = dL_di1 - dL_di0, dL/dvc = dL_di2 - dL_di0 (the reference
                        // expands the same sum over the three weights with the +-1 / 0 factors written out)
                        const float dL_duc = dL_di1 - dL_di0, dL_dvc = dL_di2 - dL_di0;
                        const float dL_du = dL_duc * duc_du + dL_dvc * dvc_du;
                        const float dL_dv = dL_duc * duc_dv + dL_dvc * dvc_dv;
                        // sufficient statistics of the vertex-position gradient (see header comment)
                        const float k1 = dL_du * inv_denom;
                        const float k24 = (dL_du * tuv.y + dL_dv * (EXACT ? tuv.z : tuv.x)) * inv_denom;
                        v[0] = k1 * rd.x; v[1] = k1 * rd.y; v[2] = k1 * rd.z;
                        v[3] = k24 * rd.x; v[4] = k24 * rd.y; v[5] = k24 * rd.z;
                        v[6] = dL_dv * inv_denom;
                        if constexpr (EXACT) {
                            const float kv = v[6];
                            v[6] = kv * rd.x; v[21] = kv * rd.y; v[22] = kv * rd.z;
                        }
                        if constexpr (CAM) {
                            const float3 p0 = f3(a0.x, a0.y, a0.z);
                            const float3 Tv = ro - p0, E1 = f3(a1.x, a1.y, a1.z) - p0, E2 = f3(a2.x, a2.y, a2.z) - p0;
                            const float kv = dL_dv * inv_denom;
                            const float kn = EXACT ? k24 : (dL_du * tuv.y + dL_dv * tuv.z) * inv_denom;
                            g_ro = g_ro + k1 * cross3(rd, E2) + kv * cross3(E1, rd);
                            g_rd = g_rd + k1 * cross3(E2, Tv) + kv * cross3(Tv, E1) - kn * cross3(E2, E1);
                        }
                    }
                }

                // ---- reduce over the two lanes of each group: 24 -> 12 values per lane; lane class c = lane & 1
                //      owns logical 12c..12c+11 = three 16-byte vectors, the c-th half of each 32-byte sector of the
                //      record (stat_slot)
                xreduce_step<12, 1>(v, h1);
                if (DET) {
                    if (have) {
                        // fixed-point record in LOGICAL order: this lane holds sums 12*cls .. 12*cls+11
                        const int cls = lane & 1;
                        long long* rec = p.det_stats + (size_t)s_rec[j * 9 + 1].w * 24 + 12 * cls;
                        const ptrdiff_t det_hi = TriDetLayout::hi_offset(p.B, p.P, p.F);
#pragma unroll
                        for (int k = 0; k < 12; k++) {
                            if (cls == 1 && k >= (EXACT ? 11 : 9)) break;        // logical 21..23 (EXACT: 23): padding
                            // vertex-position statistics: logical 0..6 (EXACT: and 21, 22) take the finer scale
                            const bool pos = cls == 0 ? k < 7 : (EXACT && k >= 9);
                            det_add(rec + k, v[k], pos ? det_sg : det_sv, det_hi, p.det_gmax);
                        }
                    }
                } else if (have) {
                    // index of the (view, face) record (staged next to the positions) and the lane class in one address
                    float* rec = stats + ((size_t)s_rec[j * 9 + 1].w * 6 + (size_t)h1) * 4;
                    red_add_v4(rec, v[0], v[1], v[2], v[3]);
                    red_add_v4(rec + 8, v[4], v[5], v[6], v[7]);
                    red_add_v4(rec + 16, v[8], v[9], v[10], v[11]);
                }
            }
            __syncwarp();   // the next pass overwrites the index list and the masks
        }
    }
    if constexpr (CAM) {
        // chain this pixel into the 24 partials: g_d = dL/dd, then d = L pv, pv = (inv_proj n).xyz, n = (nx, ny, -1, 1)
        //   [3j + i]       dL/dinv_mv[4j + i]  = g_d[i] pv[j]     (i, j < 3)
        //   [9 + i]        dL/dinv_mv[12 + i]  = g_ro[i]
        //   [12 + 3k + j]  dL/dinv_proj[4k + j] = (L^T g_d)[j] n[k]  (j < 3, k < 4)
        float g[DMR_CAM_REC];
#pragma unroll
        for (int k = 0; k < DMR_CAM_REC; k++) g[k] = 0.0f;
        if (inside) {
            const float* imv = p.inv_mv + 16 * b;
            const float* ipj = p.inv_proj + 16 * b;
            const float n[4] = { pix2ndc(px + 0.5f, p.W), pix2ndc(py + 0.5f, p.H), -1.0f, 1.0f };
            float pv[3], d[3];
#pragma unroll
            for (int j = 0; j < 3; j++) pv[j] = ipj[j] * n[0] + ipj[4 + j] * n[1] + ipj[8 + j] * n[2] + ipj[12 + j];
#pragma unroll
            for (int i = 0; i < 3; i++) d[i] = imv[i] * pv[0] + imv[4 + i] * pv[1] + imv[8 + i] * pv[2];
            const float dn = sqrtf(d[0] * d[0] + d[1] * d[1] + d[2] * d[2]);
            const float sl = dn + 0.0000001f;
            const float dg = (d[0] * g_rd.x + d[1] * g_rd.y + d[2] * g_rd.z) / (sl * sl * fmaxf(dn, 1e-30f));
            const float gd[3] = { g_rd.x / sl - d[0] * dg, g_rd.y / sl - d[1] * dg, g_rd.z / sl - d[2] * dg };
#pragma unroll
            for (int j = 0; j < 3; j++) {
#pragma unroll
                for (int i = 0; i < 3; i++) g[3 * j + i] = gd[i] * pv[j];
                const float lg = imv[4 * j] * gd[0] + imv[4 * j + 1] * gd[1] + imv[4 * j + 2] * gd[2];
#pragma unroll
                for (int k = 0; k < 4; k++) g[12 + 3 * k + j] = lg * n[k];
            }
            g[9] = g_ro.x; g[10] = g_ro.y; g[11] = g_ro.z;
        }
        // fixed-order reduction: warp butterfly, then the eight warp sums in warp order
#pragma unroll
        for (int k = 0; k < DMR_CAM_REC; k++) {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) g[k] += __shfl_xor_sync(0xffffffffu, g[k], o);
        }
        __syncthreads();                                   // s_rec is free again
        float* const s_cam = reinterpret_cast<float*>(s_rec);
        if (lane < DMR_CAM_REC) {
            float x = g[0];
#pragma unroll
            for (int k = 1; k < DMR_CAM_REC; k++) x = lane == k ? g[k] : x;
            s_cam[warp * DMR_CAM_REC + lane] = x;
        }
        __syncthreads();
        if (tid < DMR_CAM_REC) {
            float sum = 0.0f;
#pragma unroll
            for (int w = 0; w < 8; w++) sum += s_cam[w * DMR_CAM_REC + tid];
            cam_tiles[((size_t)b * tiles_x * tiles_y + blockIdx.y * tiles_x + blockIdx.x) * DMR_CAM_REC + tid] = sum;
        }
    }
}

__global__ void __launch_bounds__(256, DMR_TRI_BWD_MINB) tri_render_bwd_kernel(TriRenderParams p)
{
    griddep_wait();   // programmatic dependent launch: see dmr_launch (common.cuh)
    tri_render_bwd_body<false, false>(p, nullptr);
}

__global__ void __launch_bounds__(256, DMR_TRI_BWD_MINB) tri_render_bwd_det_kernel(TriRenderParams p)
{
    griddep_wait();   // programmatic dependent launch: see dmr_launch (common.cuh)
    tri_render_bwd_body<true, false>(p, nullptr);
}

// Camera-gradient instantiations: the same walk plus g_ro / g_rd per lane (six more live floats) and the per-tile
// record.  Resident CTAs per SM: see DESIGN.md 3.3 for the -Xptxas -v figures of both choices.
constexpr int DMR_TRI_BWD_CAM_MINB = 3;
__global__ void __launch_bounds__(256, DMR_TRI_BWD_CAM_MINB) tri_render_bwd_cam_kernel(TriRenderParams p, float* cam_tiles)
{
    griddep_wait();   // programmatic dependent launch: see dmr_launch (common.cuh)
    tri_render_bwd_body<false, true>(p, cam_tiles);
}

__global__ void __launch_bounds__(256, DMR_TRI_BWD_CAM_MINB) tri_render_bwd_cam_det_kernel(TriRenderParams p, float* cam_tiles)
{
    griddep_wait();   // programmatic dependent launch: see dmr_launch (common.cuh)
    tri_render_bwd_body<true, true>(p, cam_tiles);
}

// Exact vertex-position instantiations of the four kernels above: two more live floats per hit (kv * rd.y, kv * rd.z
// in the reduction).  Resident CTAs per SM, measured against the default kernel: 4 (64 registers, 48 bytes of spill)
// costs 1.006x at C4 and 1.003x at C2, 3 (80 registers, no spill) 1.07x / 1.05x (DESIGN.md 3.3).  The camera
// instantiations keep DMR_TRI_BWD_CAM_MINB.
constexpr int DMR_TRI_BWD_EXACT_MINB = DMR_TRI_BWD_MINB;
__global__ void __launch_bounds__(256, DMR_TRI_BWD_EXACT_MINB) tri_render_bwd_exact_kernel(TriRenderParams p)
{
    griddep_wait();   // programmatic dependent launch: see dmr_launch (common.cuh)
    tri_render_bwd_body<false, false, true>(p, nullptr);
}

__global__ void __launch_bounds__(256, DMR_TRI_BWD_EXACT_MINB) tri_render_bwd_exact_det_kernel(TriRenderParams p)
{
    griddep_wait();   // programmatic dependent launch: see dmr_launch (common.cuh)
    tri_render_bwd_body<true, false, true>(p, nullptr);
}

__global__ void __launch_bounds__(256, DMR_TRI_BWD_CAM_MINB) tri_render_bwd_exact_cam_kernel(TriRenderParams p, float* cam_tiles)
{
    griddep_wait();   // programmatic dependent launch: see dmr_launch (common.cuh)
    tri_render_bwd_body<false, true, true>(p, cam_tiles);
}

__global__ void __launch_bounds__(256, DMR_TRI_BWD_CAM_MINB) tri_render_bwd_exact_cam_det_kernel(TriRenderParams p, float* cam_tiles)
{
    griddep_wait();   // programmatic dependent launch: see dmr_launch (common.cuh)
    tri_render_bwd_body<true, true, true>(p, cam_tiles);
}

// Alpha-cotangent instantiations: the eight kernels above (default / deterministic x camera x exact) plus dL/dalpha,
// which travels as an argument of its own so that TriRenderParams stays as it is.  Resident CTAs per SM as the kernel
// each one stands in for; -Xptxas -v of all of them in DESIGN.md 3.3.
template <bool DET, bool CAM, bool EXACT>
__global__ void __launch_bounds__(256, CAM ? DMR_TRI_BWD_CAM_MINB : EXACT ? DMR_TRI_BWD_EXACT_MINB : DMR_TRI_BWD_MINB)
tri_render_bwd_alpha_kernel(TriRenderParams p, float* cam_tiles, const float* __restrict__ dL_dalpha)
{
    griddep_wait();   // programmatic dependent launch: see dmr_launch (common.cuh)
    tri_render_bwd_body<DET, CAM, EXACT, true>(p, cam_tiles, dL_dalpha);
}

template <bool DET>
static cudaError_t launch_tri_bwd_alpha(dim3 grid, cudaStream_t stream, const TriRenderParams& p, float* cam_tiles, bool exact,
                                        const float* dL_dalpha)
{
    if (cam_tiles)
        return exact ? dmr_launch(tri_render_bwd_alpha_kernel<DET, true, true>, grid, dim3(256), 0, stream, p, cam_tiles, dL_dalpha)
                     : dmr_launch(tri_render_bwd_alpha_kernel<DET, true, false>, grid, dim3(256), 0, stream, p, cam_tiles, dL_dalpha);
    float* const none = nullptr;
    return exact ? dmr_launch(tri_render_bwd_alpha_kernel<DET, false, true>, grid, dim3(256), 0, stream, p, none, dL_dalpha)
                 : dmr_launch(tri_render_bwd_alpha_kernel<DET, false, false>, grid, dim3(256), 0, stream, p, none, dL_dalpha);
}

// One CTA per view: the view's per-tile camera records (tri_render_bwd_cam_kernel) are summed in a fixed order -- a
// thread owns one component (240 = 10 x 24 threads, coalesced reads of the flat record array), then the ten partial
// sums of a component are added in thread order -- and chained through the inverses: with N = A^-1,
// dL/dA = -N^T (dL/dN) N^T.  The result is ADDED to dL_dmv[b] / dL_dproj[b]; this CTA is the only writer of view b.
__global__ void __launch_bounds__(240) tri_camera_finish_kernel(int ntiles, const float* __restrict__ cam_tiles,
                                                                const float* __restrict__ inv_mv, const float* __restrict__ inv_proj,
                                                                float* __restrict__ dL_dmv, float* __restrict__ dL_dproj)
{
    griddep_wait();   // programmatic dependent launch: see dmr_launch (common.cuh)
    __shared__ float s_part[240];
    __shared__ float s_g[2][16];      // dL/dinv_mv, dL/dinv_proj (column-major, zeros where the forward reads nothing)
    const int b = blockIdx.x, t = threadIdx.x;
    const float* rec = cam_tiles + (size_t)b * ntiles * DMR_CAM_REC;
    const size_t n = (size_t)ntiles * DMR_CAM_REC;
    float acc = 0.0f;
    for (size_t i = t; i < n; i += 240) acc += rec[i];   // component t % 24
    s_part[t] = acc;
    __syncthreads();
    if (t < 32) {
        s_g[t >> 4][t & 15] = 0.0f;
        __syncwarp();
        if (t < DMR_CAM_REC) {
            float sum = 0.0f;
#pragma unroll
            for (int k = 0; k < 10; k++) sum += s_part[t + DMR_CAM_REC * k];
            // record slot -> column-major matrix entry (cam record layout: tri_render_bwd_body)
            if (t < 9) s_g[0][4 * (t / 3) + t % 3] = sum;
            else if (t < 12) s_g[0][12 + t - 9] = sum;
            else s_g[1][4 * ((t - 12) / 3) + (t - 12) % 3] = sum;
        }
        __syncwarp();
        // thread e: entry (i, j) = (e & 3, (e >> 2) & 3) of matrix e >> 4; M(r, c) = m[4c + r]
        const int m = t >> 4, e = t & 15, i = e & 3, j = e >> 2;
        const float* N = (m == 0 ? inv_mv : inv_proj) + 16 * b;
        const float out = inverse_chain(N, s_g[m], i, j);
        float* dst = (m == 0 ? dL_dmv : dL_dproj) + 16 * b + e;
        *dst += -out;
    }
}

// Deterministic mode: g = max |dL_dout| over both cotangent images, as float bits (non-negative floats order like
// unsigned integers; the maximum does not depend on the order of the comparisons).
__global__ void __launch_bounds__(256) det_gmax_kernel(const float* __restrict__ a, size_t na, const float* __restrict__ b,
                                                           size_t nb, uint32_t* __restrict__ gmax)
{
    griddep_wait();   // programmatic dependent launch: see dmr_launch (common.cuh)
    uint32_t m = 0;
    for (size_t i = (size_t)blockIdx.x * 256 + threadIdx.x; i < na + nb; i += (size_t)gridDim.x * 256) {
        const float x = i < na ? a[i] : b[i - na];
        m = max(m, __float_as_uint(fabsf(x)));
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0 && m != 0) atomicMax(gmax, m);
}

// Once per FACE: statistics of all views -> gradients of the five inputs (see tri_render_bwd_kernel).
// One thread owns face f and walks its B statistics records (view-major, 96 B each, independent loads): the
// vertex-position and colour gradients of the views are summed in registers and scattered to the three vertices
// ONCE, the world-space triangle (48 B of the record; identical in every view's record) is read once, from view 0.
// The first version ran one thread per (view, face): at C4 (8 views per call) it re-read the triangle and
// re-scattered to the same vertices eight times -- 2.46 GB read + 0.73 GB written, HBM-bound at 520 us.
// EXACT: the statistics of tri_render_bwd_body<.., EXACT> (S3v in logical 6, 21, 22).
template <bool DET, bool MULTI, bool EXACT = false>   // MULTI = false: B == 1 (no view loop, no accumulators: 54 instead of 74 registers)
__device__ __forceinline__ void tri_grad_finish_body(const TriRenderParams& p)
{
    const int nviews = MULTI ? p.B : 1;
    const size_t f = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= (size_t)p.F) return;
    float det_sv = 0.0f, det_sg = 0.0f;
    double iv = 0.0, ig = 0.0;
    ptrdiff_t hi = 0;
    if (DET) {
        det_scales(*p.det_gmax, det_sv, det_sg);
        hi = TriDetLayout::hi_offset(p.B, p.P, p.F);
        if (det_poisoned(p.det_gmax)) {
            for (int b = 0; b < nviews; b++) p.dL_dfintense[(size_t)b * p.F + f] = __int_as_float(0x7fc00000);
            return;
        }
        if (det_sv == 0.0f) return;
        iv = 1.0 / (double)det_sv; ig = 1.0 / (double)det_sg;
    }
    bool have_tri = false;
    float3 v0 = f3(0, 0, 0), E1 = f3(0, 0, 0), E2 = f3(0, 0, 0);
    int vi[3] = { 0, 0, 0 };
    float3 dps[3] = { f3(0, 0, 0), f3(0, 0, 0), f3(0, 0, 0) };   // sum over views of dL_dp0..2
    float cs[9] = { 0, 0, 0, 0, 0, 0, 0, 0, 0 };                  // ... of dL_dcolor[3][3]
    float opa = 0.0f;                                             // ... of dL_dopacity
    for (int b = 0; b < nviews; b++) {
        const size_t idx = (size_t)b * p.F + f;
        float st[24];
        bool any = false;
        if (DET) {
            const long long* r = p.det_stats + idx * 24;
#pragma unroll
            for (int i = 0; i < (EXACT ? 23 : 21); i++) {
                any = any || det_nonzero(r + i, hi);
                st[i] = (float)det_value(r + i, hi, (i < 7 || i >= 21) ? ig : iv);
            }
            if constexpr (!EXACT) st[21] = st[22] = 0.0f;
            st[23] = 0.0f;
        } else {
            const float4* st4 = reinterpret_cast<const float4*>(p.grad_stats + idx * 24);
            float sm[24];
#pragma unroll
            for (int q = 0; q < 6; q++) {
                float4 t = st4[q];
                sm[4 * q] = t.x; sm[4 * q + 1] = t.y; sm[4 * q + 2] = t.z; sm[4 * q + 3] = t.w;
                any = any || t.x != 0.0f || t.y != 0.0f || t.z != 0.0f || t.w != 0.0f;
            }
#pragma unroll
            for (int i = 0; i < 24; i++) st[i] = sm[stat_slot(i)];
        }
        if (!any) continue;
        if (!have_tri) {
            const TriRecord* rec = p.records + f;                                   // view 0's record: bytes 28..95
            v0 = f3(rec->v0[0], rec->v0[1], rec->v0[2]);
            E1 = f3(rec->v1[0], rec->v1[1], rec->v1[2]) - v0; E2 = f3(rec->v2[0], rec->v2[1], rec->v2[2]) - v0;
            vi[0] = rec->i0; vi[1] = rec->i1; vi[2] = rec->i2;
            have_tri = true;
        }
        const float* imv = p.inv_mv + 16 * b;
        const float3 T = f3(imv[12], imv[13], imv[14]) - v0;
        const float3 S1 = f3(st[0], st[1], st[2]), S24 = f3(st[3], st[4], st[5]);
        float3 gE1, gE2, gT;
        if constexpr (EXACT) {
            const float3 S3v = f3(st[6], st[21], st[22]);
            gE1 = cross3(S3v, T) - cross3(S24, E2);
            gE2 = cross3(T, S1) - cross3(E1, S24);
            gT = cross3(S1, E2) + cross3(E1, S3v);
        } else {
            const float S3 = st[6];
            gE1 = S3 * cross3(E2, T) - cross3(S24, E2);
            gE2 = cross3(T, S1) - cross3(E1, S24) + S3 * cross3(T, E1);
            gT = cross3(S1, E2) + S3 * cross3(E1, E2);
        }
        const float3 dp[3] = { -gE1 - gE2 - gT, gE1, gE2 };
        p.dL_dfintense[idx] = st[8];
        if constexpr (DET) {
            // fixed-point accumulators: every view's terms are added as before (integer adds commute)
#pragma unroll
            for (int k = 0; k < 3; k++) {
                long long* a = p.det_vert + 8 * (size_t)vi[k];
                det_add(a + 0, dp[k].x, det_sg, hi, p.det_gmax);
                det_add(a + 1, dp[k].y, det_sg, hi, p.det_gmax);
                det_add(a + 2, dp[k].z, det_sg, hi, p.det_gmax);
                det_add(a + 4, st[12 + 3 * k], det_sv, hi, p.det_gmax);
                det_add(a + 5, st[13 + 3 * k], det_sv, hi, p.det_gmax);
                det_add(a + 6, st[14 + 3 * k], det_sv, hi, p.det_gmax);
                det_add(p.det_vdepth + (size_t)b * p.P + vi[k], st[9 + k], det_sv, hi, p.det_gmax);
            }
            det_add(p.det_fopa + f, st[7], det_sv, hi, p.det_gmax);
        } else {
#pragma unroll
            for (int k = 0; k < 3; k++) {
                dps[k] = dps[k] + dp[k];
                cs[3 * k] += st[12 + 3 * k]; cs[3 * k + 1] += st[13 + 3 * k]; cs[3 * k + 2] += st[14 + 3 * k];
                atomicAdd(p.dL_dvdepth + (size_t)b * p.P + vi[k], st[9 + k]);
            }
            opa += st[7];
        }
    }
    if constexpr (DET) return;
    if (!have_tri) return;
    // The reference scatters 6 scalar atomics per vertex and covered pixel here (backward.cu:389-407).  With many
    // faces per vertex two 16-byte vector reductions into float4-per-vertex accumulators cost a third of the
    // lane-operations (tri_grad_vertex_kernel folds them into dL_dverts / dL_dvcolor [P,3]), but the accumulators
    // are 56 B of extra streaming per VERTEX (C5, 12 M unshared vertices: 92 -> 175 us), hence the switch in
    // tri_render_backward.
    if (p.grad_vacc) {
#pragma unroll
        for (int k = 0; k < 3; k++) {
            red_add_v4(reinterpret_cast<float*>(p.grad_vacc + vi[k]), dps[k].x, dps[k].y, dps[k].z, 0.0f);
            red_add_v4(reinterpret_cast<float*>(p.grad_vacc + (size_t)p.P + vi[k]), cs[3 * k], cs[3 * k + 1], cs[3 * k + 2], 0.0f);
        }
    } else {
#pragma unroll
        for (int k = 0; k < 3; k++) {
            float* dv = p.dL_dverts + 3 * (size_t)vi[k];
            atomicAdd(dv + 0, dps[k].x); atomicAdd(dv + 1, dps[k].y); atomicAdd(dv + 2, dps[k].z);
            float* dc = p.dL_dvcolor + 3 * (size_t)vi[k];
            atomicAdd(dc + 0, cs[3 * k]); atomicAdd(dc + 1, cs[3 * k + 1]); atomicAdd(dc + 2, cs[3 * k + 2]);
        }
    }
    atomicAdd(p.dL_dfopacity + f, opa);
}

template <bool MULTI>
__global__ void __launch_bounds__(256) tri_grad_finish_kernel(TriRenderParams p) { griddep_wait(); tri_grad_finish_body<false, MULTI>(p); }
__global__ void __launch_bounds__(256) tri_grad_finish_det_kernel(TriRenderParams p) { griddep_wait(); tri_grad_finish_body<true, true>(p); }
template <bool MULTI>
__global__ void __launch_bounds__(256) tri_grad_finish_exact_kernel(TriRenderParams p) { griddep_wait(); tri_grad_finish_body<false, MULTI, true>(p); }
__global__ void __launch_bounds__(256) tri_grad_finish_exact_det_kernel(TriRenderParams p) { griddep_wait(); tri_grad_finish_body<true, true, true>(p); }

// Deterministic mode, last step: fixed-point accumulators -> += into the caller's fp32 gradient tensors.
// One thread per vertex, then per (view, vertex), then per face.
__global__ void __launch_bounds__(256) tri_det_convert_kernel(TriRenderParams p)
{
    griddep_wait();   // programmatic dependent launch: see dmr_launch (common.cuh)
    float sv, sg;
    det_scales(*p.det_gmax, sv, sg);
    const size_t P = (size_t)p.P, BP = (size_t)p.B * p.P, F = (size_t)p.F;
    size_t i = (size_t)blockIdx.x * 256 + threadIdx.x;
    if (det_poisoned(p.det_gmax)) {
        const float nan = __int_as_float(0x7fc00000);
        if (i < P) { for (int c = 0; c < 3; c++) { p.dL_dverts[3 * i + c] = nan; p.dL_dvcolor[3 * i + c] = nan; } }
        else if (i - P < BP) p.dL_dvdepth[i - P] = nan;
        else if (i - P - BP < F) p.dL_dfopacity[i - P - BP] = nan;
        return;
    }
    if (sv == 0.0f) return;
    const double iv = 1.0 / (double)sv, ig = 1.0 / (double)sg;
    const ptrdiff_t hi = TriDetLayout::hi_offset(p.B, p.P, p.F);
    if (i < P) {
        const long long* a = p.det_vert + 8 * i;
#pragma unroll
        for (int c = 0; c < 3; c++) {
            if (det_nonzero(a + c, hi)) p.dL_dverts[3 * i + c] += (float)det_value(a + c, hi, ig);
            if (det_nonzero(a + 4 + c, hi)) p.dL_dvcolor[3 * i + c] += (float)det_value(a + 4 + c, hi, iv);
        }
        return;
    }
    i -= P;
    if (i < BP) {
        const long long* a = p.det_vdepth + i;
        if (det_nonzero(a, hi)) p.dL_dvdepth[i] += (float)det_value(a, hi, iv);
        return;
    }
    i -= BP;
    if (i < F) {
        const long long* a = p.det_fopa + i;
        if (det_nonzero(a, hi)) p.dL_dfopacity[i] += (float)det_value(a, hi, iv);
    }
}

// Once per vertex: float4 accumulators -> dL_dverts[P,3], dL_dvcolor[P,3].
__global__ void __launch_bounds__(256) tri_grad_vertex_kernel(TriRenderParams p)
{
    griddep_wait();   // programmatic dependent launch: see dmr_launch (common.cuh)
    const int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= p.P) return;
    const float4 a = p.grad_vacc[v], c = p.grad_vacc[(size_t)p.P + v];
    float* dv = p.dL_dverts + 3 * (size_t)v;
    float* dc = p.dL_dvcolor + 3 * (size_t)v;
    if (a.x != 0.0f || a.y != 0.0f || a.z != 0.0f) { dv[0] += a.x; dv[1] += a.y; dv[2] += a.z; }
    if (c.x != 0.0f || c.y != 0.0f || c.z != 0.0f) { dc[0] += c.x; dc[1] += c.y; dc[2] += c.z; }
}

int tri_render_forward(const TriRenderParams& p, cudaStream_t stream)
{
    if (p.B <= 0 || p.W <= 0 || p.H <= 0) return 0;
    dim3 grid((p.W + DMR_TILE - 1) / DMR_TILE, (p.H + DMR_TILE - 1) / DMR_TILE, p.B);
    ProfScope prof(ST_TRI_FWD, stream);
    DMR_CUDA(dmr_launch(tri_render_fwd_kernel, dim3(grid), dim3(256), 0, stream, p));
    DMR_LAUNCH_CHECK("tri_render_fwd_kernel");
    return 0;
}

int tri_render_backward(const TriRenderParams& p, cudaStream_t stream, float* cam_tiles, bool exact, const float* dL_dalpha)
{
    if (p.B <= 0 || p.W <= 0 || p.H <= 0) return 0;
    dim3 grid((p.W + DMR_TILE - 1) / DMR_TILE, (p.H + DMR_TILE - 1) / DMR_TILE, p.B);
    if (dL_dalpha) {
        ProfScope prof(ST_TRI_BWD_ALPHA, stream);
        DMR_CUDA(launch_tri_bwd_alpha<false>(grid, stream, p, cam_tiles, exact, dL_dalpha));
        DMR_LAUNCH_CHECK("tri_render_bwd_alpha_kernel");
    } else if (cam_tiles) {
        ProfScope prof(ST_TRI_BWD_CAM, stream);
        DMR_CUDA(dmr_launch(exact ? tri_render_bwd_exact_cam_kernel : tri_render_bwd_cam_kernel, dim3(grid), dim3(256), 0,
                            stream, p, cam_tiles));
        DMR_LAUNCH_CHECK("tri_render_bwd_cam_kernel");
    } else {
        ProfScope prof(ST_TRI_BWD, stream);
        DMR_CUDA(dmr_launch(exact ? tri_render_bwd_exact_kernel : tri_render_bwd_kernel, dim3(grid), dim3(256), 0, stream, p));
        DMR_LAUNCH_CHECK("tri_render_bwd_kernel");
    }
    {
        ProfScope prof(ST_TRI_BWD_FINISH, stream);
        const dim3 fgrid((unsigned)((p.F + 255) / 256));
        if (p.B > 1) DMR_CUDA(dmr_launch(exact ? tri_grad_finish_exact_kernel<true> : tri_grad_finish_kernel<true>, fgrid, dim3(256), 0, stream, p));
        else DMR_CUDA(dmr_launch(exact ? tri_grad_finish_exact_kernel<false> : tri_grad_finish_kernel<false>, fgrid, dim3(256), 0, stream, p));
        DMR_LAUNCH_CHECK("tri_grad_finish_kernel");
        if (p.grad_vacc) {
            count_launch(1);   // two kernels under one scope
            DMR_CUDA(dmr_launch(tri_grad_vertex_kernel, dim3((unsigned)((p.P + 255) / 256)), dim3(256), 0, stream, p));
            DMR_LAUNCH_CHECK("tri_grad_vertex_kernel");
        }
    }
    return 0;
}

int det_gmax(const float* a, size_t na, const float* b, size_t nb, uint32_t* gmax, cudaStream_t stream)
{
    DMR_CUDA(dmr_launch(det_gmax_kernel, dim3(592), dim3(256), 0, stream, a, na, b, nb, gmax));
    DMR_LAUNCH_CHECK("det_gmax_kernel");
    return 0;
}

int tri_render_backward_deterministic(const TriRenderParams& p, cudaStream_t stream, float* cam_tiles, bool exact,
                                      const float* dL_dalpha)
{
    if (p.B <= 0 || p.W <= 0 || p.H <= 0) return 0;
    dim3 grid((p.W + DMR_TILE - 1) / DMR_TILE, (p.H + DMR_TILE - 1) / DMR_TILE, p.B);
    const size_t HW = (size_t)p.W * p.H;
    {
        ProfScope prof(dL_dalpha ? ST_TRI_BWD_ALPHA : cam_tiles ? ST_TRI_BWD_CAM : ST_TRI_BWD, stream);
        count_launch(1);   // two kernels under one scope
        int rc = det_gmax(p.dL_dcolor, 3 * p.B * HW, p.dL_ddepth, p.B * HW, const_cast<uint32_t*>(p.det_gmax), stream);
        if (rc) return rc;
        if (dL_dalpha) {
            // the fixed-point scale covers max |dL_dalpha| too: a second maximum into the same word (order-independent)
            count_launch(1);
            if ((rc = det_gmax(dL_dalpha, p.B * HW, nullptr, 0, const_cast<uint32_t*>(p.det_gmax), stream))) return rc;
            DMR_CUDA(launch_tri_bwd_alpha<true>(grid, stream, p, cam_tiles, exact, dL_dalpha));
            DMR_LAUNCH_CHECK("tri_render_bwd_alpha_det_kernel");
        } else if (cam_tiles) {
            DMR_CUDA(dmr_launch(exact ? tri_render_bwd_exact_cam_det_kernel : tri_render_bwd_cam_det_kernel, dim3(grid),
                                dim3(256), 0, stream, p, cam_tiles));
            DMR_LAUNCH_CHECK("tri_render_bwd_cam_det_kernel");
        } else {
            DMR_CUDA(dmr_launch(exact ? tri_render_bwd_exact_det_kernel : tri_render_bwd_det_kernel, dim3(grid), dim3(256), 0,
                                stream, p));
            DMR_LAUNCH_CHECK("tri_render_bwd_det_kernel");
        }
    }
    {
        ProfScope prof(ST_TRI_BWD_FINISH, stream);
        count_launch(1);
        DMR_CUDA(dmr_launch(exact ? tri_grad_finish_exact_det_kernel : tri_grad_finish_det_kernel,
                            dim3((unsigned)((p.F + 255) / 256)), dim3(256), 0, stream, p));
        DMR_LAUNCH_CHECK("tri_grad_finish_det_kernel");
        const size_t n = (size_t)p.P + (size_t)p.B * p.P + (size_t)p.F;
        DMR_CUDA(dmr_launch(tri_det_convert_kernel, dim3((unsigned)((n + 255) / 256)), dim3(256), 0, stream, p));
        DMR_LAUNCH_CHECK("tri_det_convert_kernel");
    }
    return 0;
}

int tri_camera_finish(int B, int W, int H, const float* cam_tiles, const float* inv_mv, const float* inv_proj, float* dL_dmv,
                      float* dL_dproj, cudaStream_t stream)
{
    if (B <= 0 || W <= 0 || H <= 0) return 0;
    const int ntiles = ((W + DMR_TILE - 1) / DMR_TILE) * ((H + DMR_TILE - 1) / DMR_TILE);
    ProfScope prof(ST_TRI_CAM_FINISH, stream);
    DMR_CUDA(dmr_launch(tri_camera_finish_kernel, dim3(B), dim3(240), 0, stream, ntiles, cam_tiles, inv_mv, inv_proj, dL_dmv, dL_dproj));
    DMR_LAUNCH_CHECK("tri_camera_finish_kernel");
    return 0;
}

}  // namespace dmr
