// radix_sort.cu -- hand-written onesweep LSD radix sort of (u64 key, u32 value)
// pairs on bits [0, end_bit).  Replaces cub::DeviceRadixSort::SortPairs
// (cuda_rasterizer/rasterizer_impl.cu:319-324, cuda_renderer/renderer_impl.cu:335-340).
// The result is fully specified (stable ascending order on the selected bits),
// so it is bit-identical to CUB's.
//
// Structure (per sort):
//   1. hist_kernel     one read of the keys -> all per-pass 256-bin histograms
//   2. plan_kernel     exclusive scan of each histogram; passes whose digit is
//                      constant over all keys are skipped (identity permutation);
//                      ping-pong buffers are assigned so that the LAST executed
//                      pass writes the caller's output arrays
//   3. onesweep_kernel one launch per pass: tile-local stable ranking with
//                      warp multi-split, decoupled look-back across tiles for the
//                      per-digit global prefix, scatter through shared memory so
//                      global stores are coalesced per digit run.
// Algorithmic bytes: 8 B/key (histogram) + 24 B/key per executed pass.
#include "radix_sort.cuh"

namespace dmr {

// Tile shape of a onesweep pass: threads per CTA, keys per thread, resident CTAs per SM (register cap).
// Measured on B200 after the ranking loop was tightened (one pass over the 32.1 M (u32, u32) pairs of C5, 514 MB;
// CUB's SM100 onesweep on the same pairs, same box: 279 us, tools/sort_vs_cub.cu):
//     512 x  8, 2 CTAs/SM (round 1)  250 us        256 x 16, 3 CTAs (80 regs)   205 us
//     256 x  8, 4 or 6 CTAs          287 us        256 x 16, 4 CTAs (64 regs)   193 us   <- default
//     384 x  8, 3 CTAs               248 us        256 x 20, 3 CTAs             187 us
//     512 x  8, 3 CTAs (40 regs)     232 us        512 x 16, 2 CTAs             187 us
//     512 x 16, 1 CTA (124 regs)     246 us        256 x 24 / 32, 2 CTAs        205 / 207 us (spills)
// More keys per thread amortise the per-tile work (256-digit scan, look-back, three barriers); the 4096-key tile is
// kept because the 5120 / 8192-key shapes cost 20 % on the small face sorts (C1: 30 -> 36 us).
constexpr int DMR_RS_THREADS = 256;
constexpr int DMR_RS_KPT = 16;
constexpr int DMR_RS_MINB = 4;
constexpr int RS_TILE_KEYS = DMR_RS_THREADS * DMR_RS_KPT;
#define RS_MIN_TILE 2048   // the descriptor array is sized for tiles of at least this many keys
// Small sorts (the face / tile sorts of C1, C2) are a handful of tiles on an otherwise idle GPU: a pass lasts as long as
// ONE tile takes (16 serial ranking rounds, ~6 us), not as long as the data takes to move.  Up to RS_SMALL_N keys the
// tiles are 256 x RS_SMALL_KPT keys: four times as many CTAs, a quarter of the serial rounds each.
// (Measured and rejected for these sizes: 32 instead of 8 descriptors per look-back step -- the walk over the
// predecessors is not what a small pass waits for.  And for the large shape: key and value through shared memory as
// one 64-bit word, one STS.64 / LDS.64 per pair: C5 pass 182.7 -> 186.8 us.)
constexpr unsigned RS_SMALL_N = 1u << 20;
constexpr int RS_SMALL_KPT = 8;
constexpr int RS_SMALL_TILE = 256 * RS_SMALL_KPT;
__host__ __device__ constexpr size_t rs_tile_keys(size_t n) { return n <= RS_SMALL_N ? (size_t)RS_SMALL_TILE : (size_t)RS_TILE_KEYS; }
static_assert(DMR_RS_THREADS >= 256 && DMR_RS_THREADS % 32 == 0 && RS_TILE_KEYS >= RS_MIN_TILE, "onesweep tile shape");
constexpr int RS_LB = 8;         // look-back descriptors fetched per step (C5 pass: 8 -> 180 us, 16 -> 185 us, 32 -> 186 us)

#define RS_FLAG_AGG  (1u << 30)
#define RS_FLAG_INCL (2u << 30)
#define RS_VAL_MASK  ((1u << 30) - 1u)

struct SortTempLayout {   // zeroed part first, so that a caller can merge the memset with a neighbouring one
    size_t hist, ctl, desc, zero_end_base, keys_tmp, vals_tmp, total;
    size_t ntile;
    __host__ static SortTempLayout make(size_t n, size_t key_bytes)
    {
        SortTempLayout L;
        L.ntile = n <= RS_SMALL_N ? (n + RS_SMALL_TILE - 1) / RS_SMALL_TILE : (n + RS_MIN_TILE - 1) / RS_MIN_TILE;
        size_t o = 0;
        L.hist = o;     o = align_up(o + 4 * 256 * RS_MAX_PASS, 256);
        L.ctl = o;      o = align_up(o + sizeof(SortCtl), 256);
        L.desc = o;     o = align_up(o + 4 * 256 * L.ntile * RS_MAX_PASS, 256);
        L.zero_end_base = o;
        L.keys_tmp = o; o = align_up(o + key_bytes * n, 256);
        L.vals_tmp = o; o = align_up(o + 4 * n, 256);
        L.total = o + 256;
        return L;
    }
    // bytes from the start of the buffer that must be zero before a sort of npass passes
    size_t zero_bytes(size_t n, int npass) const { return desc + 4 * 256 * ((n + rs_tile_keys(n) - 1) / rs_tile_keys(n)) * (size_t)npass; }
};

size_t sort_temp_bytes(size_t n) { return SortTempLayout::make(n, 8).total; }
size_t sort_temp_bytes_u32(size_t n) { return SortTempLayout::make(n, 4).total; }

// ---------------------------------------------------------------------------
// 1. histograms of all passes in one sweep.  8 keys per thread are loaded
// before any is consumed (memory-level parallelism); a digit that is equal for
// all 256 keys of a warp batch (the top depth byte, the batch bits, usually the
// upper tile bits) costs one shared atomic instead of 256.
// ---------------------------------------------------------------------------
#define RSH_KPT 8
template <typename KeyT>
__global__ void __launch_bounds__(256) rs_hist_kernel(const KeyT* __restrict__ keys, size_t n_cap, int npass, int end_bit,
                                                      uint32_t* __restrict__ hist, const uint32_t* __restrict__ n_dev)
{
    griddep_wait();   // programmatic dependent launch: see dmr_launch (common.cuh)
    const size_t n = rs_count((uint32_t)n_cap, n_dev);
    __shared__ uint32_t s_hist[RS_MAX_PASS * 256];
    const int tid = threadIdx.x, lane = tid & 31;
    for (int i = tid; i < npass * 256; i += 256) s_hist[i] = 0;
    __syncthreads();

    const size_t chunk = 256 * RSH_KPT;
    for (size_t base = (size_t)blockIdx.x * chunk; base < n; base += (size_t)gridDim.x * chunk) {
        KeyT k[RSH_KPT];
        const bool full = base + chunk <= n;
#pragma unroll
        for (int i = 0; i < RSH_KPT; i++) {
            size_t idx = base + (size_t)i * 256 + tid;
            k[i] = (full || idx < n) ? keys[idx] : 0;
        }
        for (int p = 0; p < npass; p++) {
            const int shift = 8 * p;
            const uint32_t mask = (end_bit - shift >= 8) ? 0xffu : ((1u << (end_bit - shift)) - 1u);
            uint32_t d[RSH_KPT];
            bool same = full;
#pragma unroll
            for (int i = 0; i < RSH_KPT; i++) {
                d[i] = (uint32_t)(k[i] >> shift) & mask;
                same = same && d[i] == d[0];
            }
            const uint32_t d0 = __shfl_sync(0xffffffffu, d[0], 0);
            if (__all_sync(0xffffffffu, same && d[0] == d0)) {
                if (lane == 0) atomicAdd(&s_hist[p * 256 + d0], 32u * RSH_KPT);
            } else {
#pragma unroll
                for (int i = 0; i < RSH_KPT; i++)
                    if (full || base + (size_t)i * 256 + tid < n) atomicAdd(&s_hist[p * 256 + d[i]], 1u);
            }
        }
    }
    __syncthreads();
    for (int i = tid; i < npass * 256; i += 256) {
        uint32_t c = s_hist[i];
        if (c) atomicAdd(&hist[i], c);
    }
}

// ---------------------------------------------------------------------------
// 2. plan: exclusive scans + pass skipping + buffer assignment (1 block)
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256) rs_plan_kernel(uint32_t* __restrict__ hist, SortCtl* __restrict__ ctl, size_t n,
                                                      int npass, const uint32_t* __restrict__ n_dev)
{
    griddep_wait();   // programmatic dependent launch: see dmr_launch (common.cuh)
    __shared__ uint32_t s_scan[256];
    __shared__ uint32_t s_skip[RS_MAX_PASS];
    rs_plan_block(hist, ctl, rs_count((uint32_t)n, n_dev), npass, s_scan, s_skip);
}

// ---------------------------------------------------------------------------
// 3. one onesweep pass
// ---------------------------------------------------------------------------
template <typename KeyT>
struct RsBuffers {
    const KeyT* kin; const uint32_t* vin;
    KeyT* kout; uint32_t* vout;
    KeyT* ktmp; uint32_t* vtmp;
};

// Lanes of the warp whose digit equals this lane's: one ballot per digit bit.  Written in PTX so that every bit
// costs four instructions (test, vote, conditional complement, and); the C++ form `bit ? m : ~m` compiled to
// seven (shift, mask, compare, vote, test, select, and-merge), and the ranking loop was 54 % of the pass.
template <int NBITS>
__device__ __forceinline__ unsigned digit_peers(uint32_t d, unsigned peers)
{
#pragma unroll
    for (int bit = 0; bit < NBITS; bit++) {
        asm("{\n\t.reg .pred p;\n\t.reg .b32 m;\n\t"
            "setp.ne.u32 p, %1, 0;\n\t"
            "vote.sync.ballot.b32 m, p, 0xffffffff;\n\t"
            "@!p not.b32 m, m;\n\t"
            "and.b32 %0, %0, m;\n\t}"
            : "+r"(peers) : "r"(d & (1u << bit)));
    }
    return peers;
}

// Phase order per tile (4096 keys, 256 threads x 16 keys):
//   load -> per-warp digit COUNTS (shared atomics) -> publish the tile aggregate EARLY -> stable
//   ranking (ballot multi-split) -> scatter into shared memory -> look-back -> coalesced write-out.
// Publishing the aggregate before the long, variable-latency ranking phase means that by the time a
// tile looks back every predecessor's aggregate is already there (no spinning on slow neighbours;
// measured: waiting at the look-back was ~35% of all stall samples when the aggregate was published
// after ranking), and the look-back only has to walk over the few predecessors that have not yet
// published their inclusive prefix -- RS_LB descriptors are fetched per step so that walk costs one
// L2 round trip per RS_LB tiles.
// NBITS = digit bits of this pass (8 except for the top pass of a sort): a compile-time constant so that the
// ranking loop is exactly NBITS ballots with no run-time tests.
// FULL = every key slot of the tile is valid (all tiles of a pass but the last): no bounds tests, no padding class.
template <typename KeyT, int RS_THREADS, int RS_KPT, int NBITS, bool FULL>
__device__ __forceinline__ void rs_onesweep_tile(const RsBuffers<KeyT>& buf, size_t n, int pass,
                                                 const uint32_t* __restrict__ hist_excl, SortCtl* __restrict__ ctl,
                                                 uint32_t* __restrict__ desc, unsigned char* rs_smem, uint32_t tile,
                                                 uint32_t* s_wsum)
{
    constexpr int RS_TILE = RS_THREADS * RS_KPT;
    constexpr int RS_WARPS = RS_THREADS / 32;
    KeyT* s_keys = reinterpret_cast<KeyT*>(rs_smem);                               // RS_TILE
    uint32_t* s_vals = reinterpret_cast<uint32_t*>(rs_smem + sizeof(KeyT) * RS_TILE);   // RS_TILE
    uint32_t* s_whist = s_vals + RS_TILE;                                          // RS_WARPS * 256
    uint32_t* s_dbase = s_whist + RS_WARPS * 256;                                  // 256: local exclusive digit base
    int32_t*  s_gbase = reinterpret_cast<int32_t*>(s_dbase + 256);                 // 256: global pos - local pos (wrapping)

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t s = ctl->src[pass], d_sel = ctl->dst[pass];
    const KeyT* kin = (s == 0) ? buf.kin : (s == 1 ? buf.kout : buf.ktmp);
    const uint32_t* vin = (s == 0) ? buf.vin : (s == 1 ? buf.vout : buf.vtmp);   // buf.vin may be null: identity
    KeyT* kout = (d_sel == 1) ? buf.kout : buf.ktmp;
    uint32_t* vout = (d_sel == 1) ? buf.vout : buf.vtmp;

    const size_t tile_base = (size_t)tile * RS_TILE;
    const uint32_t nvalid = FULL ? (uint32_t)RS_TILE : (uint32_t)(n - tile_base);

    const int shift = 8 * pass;
    constexpr uint32_t dmask = (1u << NBITS) - 1u;

    // warp-striped load: item i of lane l sits at warp_base + i*32 + l, so that
    // (i, lane) order == global order (stability)
    const uint32_t wbase = warp * (32 * RS_KPT);
    KeyT key[RS_KPT];
    uint32_t val[RS_KPT];
#pragma unroll
    for (int i = 0; i < RS_KPT; i++) {
        uint32_t loc = wbase + i * 32 + lane;
        key[i] = (FULL || loc < nvalid) ? kin[tile_base + loc] : (KeyT)~(KeyT)0;
    }
    if (vin) {
#pragma unroll
        for (int i = 0; i < RS_KPT; i++) {
            uint32_t loc = wbase + i * 32 + lane;
            val[i] = (FULL || loc < nvalid) ? vin[tile_base + loc] : 0u;
        }
    } else {   // null = identity
#pragma unroll
        for (int i = 0; i < RS_KPT; i++) val[i] = (uint32_t)(tile_base + wbase + i * 32 + lane);
    }

    // ---- per-warp digit counts
    uint32_t* wh = s_whist + warp * 256;
    uint32_t dig[RS_KPT];
#pragma unroll
    for (int i = 0; i < RS_KPT; i++) {
        uint32_t loc = wbase + i * 32 + lane;
        dig[i] = (uint32_t)(key[i] >> shift) & dmask;
        if (FULL || loc < nvalid) atomicAdd(&wh[dig[i]], 1u);
    }
    __syncthreads();

    // ---- thread t < 256 owns digit t: exclusive scan over warps, tile count, EARLY publication
    uint32_t count = 0;
    uint32_t* my_desc = nullptr;
    uint32_t incl = 0;
    if (tid < 256) {
#pragma unroll
        for (int w = 0; w < RS_WARPS; w++) {
            uint32_t t = s_whist[w * 256 + tid];
            s_whist[w * 256 + tid] = count;      // becomes the warp's running write offset for this digit
            count += t;
        }
        my_desc = desc + ((size_t)pass * gridDim.x + tile) * 256 + tid;
        st_volatile_u32(my_desc, (tile == 0 ? RS_FLAG_INCL : RS_FLAG_AGG) | count);
        // exclusive scan over digits (local base inside the tile)
        incl = count;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t;
        }
        if (lane == 31) s_wsum[warp] = incl;
    }
    __syncthreads();
    if (tid < 256) {
        uint32_t woff = 0;
#pragma unroll
        for (int w = 0; w < 8; w++) if (w < warp) woff += s_wsum[w];
        s_dbase[tid] = woff + incl - count;
    }
    __syncthreads();

    // ---- stable rank inside the warp (running per-warp offsets), scatter into shared memory.
    //      One round per key of the thread: digit_peers gives the lanes holding the same digit (padding lanes of a
    //      partial tile form a class of their own), the lowest of them advances the warp's running offset for that
    //      digit, and each lane scatters to digit base + offset + its rank among the peers.
    //      (Measured and rejected: packed per-round counters -- 8 x 8-bit counts per (warp, digit) filled by the
    //      leader of every digit run, ranks from byte prefixes -- which make the 8 rounds independent of each
    //      other: 306 vs 282 us per pass at C5; the extra shared-memory traffic costs more than the chain.
    //      A single match.any.sync per key instead of the ballots: 9 % slower, its issue rate is far lower.
    //      Ranking BEFORE the scan, so that the per-warp counts fall out of the ballots and the 16 counting atomics per
    //      thread disappear (ranks parked in registers as 16-bit pairs, values loaded after the ranking): C5 pass
    //      182.7 -> 182.7 us, C4 105 / 99 -> 107 / 103 us, face sorts +2..6 % -- the aggregate is published a ranking
    //      phase later and the successors' look-back waits for it; the atomics were not what the pass waits for.)
    const uint32_t lt_mask = (1u << lane) - 1u;
#pragma unroll
    for (int i = 0; i < RS_KPT; i++) {
        const bool ok = FULL || wbase + i * 32 + lane < nvalid;
        const uint32_t d = dig[i];
        unsigned pr = 0xffffffffu;
        if (!FULL) { pr = __ballot_sync(0xffffffffu, ok); if (!ok) pr = ~pr; }
        pr = digit_peers<NBITS>(d, pr);
        const int leader = __ffs(pr) - 1;
        const uint32_t before = __popc(pr & lt_mask);
        uint32_t old = 0;
        if (ok && lane == leader) { old = wh[d]; wh[d] = old + __popc(pr); }
        old = __shfl_sync(0xffffffffu, old, leader);
        if (ok) {
            uint32_t pos = s_dbase[d] + old + before;
            s_keys[pos] = key[i];
            s_vals[pos] = val[i];
        }
        __syncwarp();
    }

    // ---- decoupled look-back for digit `tid`: sum the aggregates of the predecessors back to the nearest
    //      inclusive prefix.  RS_LB descriptors are fetched per step (one L2 round trip) and consumed WITHOUT
    //      branches: "all ready" is one unsigned minimum over the words (a flag of 0 makes the word < RS_FLAG_AGG),
    //      the running predicate `open` (no inclusive prefix seen yet) masks the additions.  ~5 instructions per
    //      descriptor; the first form (a bounds test, a spin loop and two branches per descriptor, 64-bit address
    //      arithmetic per load) cost ~25 and the look-back was 29 % of the instructions of a pass at C5 (46
    //      descriptors walked per tile and digit on average).
    if (tid < 256) {
        uint32_t excl = 0;
        if (tile > 0) {
            const uint32_t* bp = desc + ((size_t)pass * gridDim.x + (tile - 1)) * 256 + tid;   // tile - 1, then backwards
            uint32_t left = tile;              // predecessors not yet consumed (tile 0 always holds an inclusive prefix)
            bool open = true;
            while (open) {
                if (left >= RS_LB) {
                    uint32_t v[RS_LB];
#pragma unroll
                    for (int i = 0; i < RS_LB; i++) v[i] = ld_volatile_u32(bp - i * 256);
                    uint32_t mn = v[0];
#pragma unroll
                    for (int i = 1; i < RS_LB; i++) mn = min(mn, v[i]);
                    if (mn < RS_FLAG_AGG) continue;              // a predecessor has not published yet: fetch again
#pragma unroll
                    for (int i = 0; i < RS_LB; i++) {
                        excl += open ? (v[i] & RS_VAL_MASK) : 0u;
                        open = open && v[i] < RS_FLAG_INCL;
                    }
                    bp -= RS_LB * 256;
                    left -= RS_LB;
                } else {                                         // the first RS_LB tiles of a pass: one predicated batch
                    uint32_t v[RS_LB];                           // (slots beyond tile 0 read as an empty inclusive prefix)
#pragma unroll
                    for (int i = 0; i < RS_LB; i++) v[i] = (uint32_t)i < left ? ld_volatile_u32(bp - i * 256) : RS_FLAG_INCL;
                    uint32_t mn = v[0];
#pragma unroll
                    for (int i = 1; i < RS_LB; i++) mn = min(mn, v[i]);
                    if (mn < RS_FLAG_AGG) continue;
#pragma unroll
                    for (int i = 0; i < RS_LB; i++) {
                        excl += open ? (v[i] & RS_VAL_MASK) : 0u;
                        open = open && v[i] < RS_FLAG_INCL;
                    }
                    // tile 0 holds an inclusive prefix, so the walk has ended (open == false)
                }
            }
            st_volatile_u32(my_desc, RS_FLAG_INCL | (excl + count));
        }
        s_gbase[tid] = (int32_t)(hist_excl[pass * 256 + tid] + excl - s_dbase[tid]);
    }
    __syncthreads();

    // ---- coalesced write-out
    if (FULL) {
#pragma unroll
        for (int i = 0; i < RS_KPT; i++) {
            const uint32_t p = i * RS_THREADS + tid;
            KeyT k = s_keys[p];
            uint32_t d = (uint32_t)(k >> shift) & dmask;
            size_t g = (size_t)(uint32_t)(s_gbase[d] + (int32_t)p);
            kout[g] = k;
            vout[g] = s_vals[p];
        }
    } else {
        for (uint32_t p = tid; p < nvalid; p += RS_THREADS) {
            KeyT k = s_keys[p];
            uint32_t d = (uint32_t)(k >> shift) & dmask;
            size_t g = (size_t)(uint32_t)(s_gbase[d] + (int32_t)p);
            kout[g] = k;
            vout[g] = s_vals[p];
        }
    }
}

template <typename KeyT, int RS_THREADS, int RS_KPT, int RS_MINB, int NBITS>
__global__ void __launch_bounds__(RS_THREADS, RS_MINB) rs_onesweep_kernel(RsBuffers<KeyT> buf, size_t n_cap, int pass,
                                                                          const uint32_t* __restrict__ hist_excl,
                                                                          SortCtl* __restrict__ ctl, uint32_t* __restrict__ desc,
                                                                          const uint32_t* __restrict__ n_dev)
{
    griddep_wait();   // programmatic dependent launch: see dmr_launch (common.cuh)
    constexpr int RS_TILE = RS_THREADS * RS_KPT;
    constexpr int RS_WARPS = RS_THREADS / 32;
    if (!ctl->exec[pass]) return;
    // the grid is sized for the buffers' capacity; with the count on the device the CTAs beyond it leave at once
    // (tickets are handed out in launch order, so the tiles that do exist are 0 .. ceil(n / RS_TILE) - 1)
    const size_t n = rs_count((uint32_t)n_cap, n_dev);
    extern __shared__ __align__(16) unsigned char rs_smem[];
    __shared__ uint32_t s_tile;
    __shared__ uint32_t s_wsum[8];
    uint32_t* s_whist = reinterpret_cast<uint32_t*>(rs_smem + sizeof(KeyT) * RS_TILE) + RS_TILE;
    const int tid = threadIdx.x;
    if (tid == 0) s_tile = atomicAdd(&ctl->ticket[pass], 1u);
    for (int i = tid; i < RS_WARPS * 256; i += RS_THREADS) s_whist[i] = 0;
    __syncthreads();
    const uint32_t tile = s_tile;
    if ((size_t)tile * RS_TILE >= n) return;
    if ((size_t)(tile + 1) * RS_TILE <= n)
        rs_onesweep_tile<KeyT, RS_THREADS, RS_KPT, NBITS, true>(buf, n, pass, hist_excl, ctl, desc, rs_smem, tile, s_wsum);
    else
        rs_onesweep_tile<KeyT, RS_THREADS, RS_KPT, NBITS, false>(buf, n, pass, hist_excl, ctl, desc, rs_smem, tile, s_wsum);
}

template <typename KeyT, int THREADS, int KPT, int MINB>
static int launch_onesweep(const RsBuffers<KeyT>& buf, size_t n, int npass, int end_bit, const uint32_t* hist, SortCtl* ctl,
                           uint32_t* desc, bool profile, cudaStream_t stream, const uint32_t* n_dev)
{
    constexpr size_t tile = (size_t)THREADS * KPT;
    constexpr size_t smem = sizeof(KeyT) * tile + 4 * tile + 4 * (THREADS / 32) * 256 + 4 * 256 + 4 * 256;
    typedef void (*Kern)(RsBuffers<KeyT>, size_t, int, const uint32_t*, SortCtl*, uint32_t*, const uint32_t*);
    static const Kern kern[8] = {
        rs_onesweep_kernel<KeyT, THREADS, KPT, MINB, 1>, rs_onesweep_kernel<KeyT, THREADS, KPT, MINB, 2>,
        rs_onesweep_kernel<KeyT, THREADS, KPT, MINB, 3>, rs_onesweep_kernel<KeyT, THREADS, KPT, MINB, 4>,
        rs_onesweep_kernel<KeyT, THREADS, KPT, MINB, 5>, rs_onesweep_kernel<KeyT, THREADS, KPT, MINB, 6>,
        rs_onesweep_kernel<KeyT, THREADS, KPT, MINB, 7>, rs_onesweep_kernel<KeyT, THREADS, KPT, MINB, 8> };
    static bool attr_set[64] = {};   // function attributes are per device
    int dev = 0;
    DMR_CUDA(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 64 || !attr_set[dev]) {
        for (int i = 0; i < 8; i++)
            DMR_CUDA(cudaFuncSetAttribute(kern[i], cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        if (dev >= 0 && dev < 64) attr_set[dev] = true;
    }
    const unsigned ntile = (unsigned)((n + tile - 1) / tile);
    for (int p = 0; p < npass; p++) {
        const int nbits = (end_bit - 8 * p >= 8) ? 8 : (end_bit - 8 * p);
        if (profile) prof_begin(ST_SORT_PASS0 + p, stream); else count_launch(1);
        DMR_CUDA(dmr_launch(kern[nbits - 1], dim3(ntile), dim3(THREADS), smem, stream, buf, n, p, hist, ctl, desc, n_dev));
        if (profile) prof_end(ST_SORT_PASS0 + p, stream);
        DMR_LAUNCH_CHECK("rs_onesweep_kernel");
    }
    return 0;
}

// profile == false: the kernels are counted but get no stage events of their own (the face sort is reported as
// ONE stage by its caller; the per-kernel stages belong to the instance sort).
// prehist == true: the producer of the keys has already zeroed the control region (sort_pre_begin), accumulated
// the histograms and computed the plan (radix_sort.cuh); only the passes run here.
template <typename KeyT>
static int sort_pairs_impl(const KeyT* keys_in, const uint32_t* vals_in, KeyT* keys_out, uint32_t* vals_out, size_t n,
                           int end_bit, void* temp, bool profile, int prehist /* 0 no, 1 yes, 2 zeroed only */, cudaStream_t stream,
                           const uint32_t* n_dev = nullptr)
{
    if (n == 0) return 0;
    if (end_bit < 1 || end_bit > (int)(8 * sizeof(KeyT))) { set_error("sort_pairs: end_bit %d out of range", end_bit); return 1; }
    if (n >= (1ull << 30)) { set_error("sort_pairs: n=%zu exceeds 2^30", n); return 3; }
    const int npass = (end_bit + 7) / 8;
    SortTempLayout L = SortTempLayout::make(n, sizeof(KeyT));
    unsigned char* t = static_cast<unsigned char*>(temp);
    uint32_t* hist = reinterpret_cast<uint32_t*>(t + L.hist);
    SortCtl* ctl = reinterpret_cast<SortCtl*>(t + L.ctl);
    uint32_t* desc = reinterpret_cast<uint32_t*>(t + L.desc);

    static int sm_count = 0;
    if (sm_count == 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, dev);
        if (sm_count <= 0) sm_count = 148;
    }
    if (prehist != 1) {
        if (prehist == 0) DMR_CUDA(cudaMemsetAsync(t, 0, L.zero_bytes(n, npass), stream));
        size_t hblocks = (n + 256 * RSH_KPT - 1) / (256 * RSH_KPT);
        size_t hmax = (size_t)sm_count * 8;   // 8 resident CTAs per SM
        if (hblocks > hmax) hblocks = hmax;
        {
            if (profile) prof_begin(ST_SORT_HIST, stream); else count_launch(1);
            DMR_CUDA(dmr_launch(rs_hist_kernel<KeyT>, dim3((unsigned)hblocks), dim3(256), 0, stream, keys_in, n, npass, end_bit, hist, n_dev));
            if (profile) prof_end(ST_SORT_HIST, stream);
            DMR_LAUNCH_CHECK("rs_hist_kernel");
        }
        {
            if (profile) prof_begin(ST_SORT_PLAN, stream); else count_launch(1);
            DMR_CUDA(dmr_launch(rs_plan_kernel, dim3(1), dim3(256), 0, stream, hist, ctl, n, npass, n_dev));
            if (profile) prof_end(ST_SORT_PLAN, stream);
            DMR_LAUNCH_CHECK("rs_plan_kernel");
        }
    }
    RsBuffers<KeyT> buf;
    buf.kin = keys_in; buf.vin = vals_in; buf.kout = keys_out; buf.vout = vals_out;
    buf.ktmp = reinterpret_cast<KeyT*>(t + L.keys_tmp);
    buf.vtmp = reinterpret_cast<uint32_t*>(t + L.vals_tmp);
    if (n <= RS_SMALL_N)
        return launch_onesweep<KeyT, 256, RS_SMALL_KPT, 4>(buf, n, npass, end_bit, hist, ctl, desc, profile, stream, n_dev);
    return launch_onesweep<KeyT, DMR_RS_THREADS, DMR_RS_KPT, DMR_RS_MINB>(buf, n, npass, end_bit, hist, ctl, desc, profile, stream, n_dev);
}

int sort_pairs(const uint64_t* keys_in, const uint32_t* vals_in, uint64_t* keys_out, uint32_t* vals_out, size_t n,
               int end_bit, void* temp, cudaStream_t stream)
{
    return sort_pairs_impl<uint64_t>(keys_in, vals_in, keys_out, vals_out, n, end_bit, temp, true, 0, stream);
}

int sort_pairs_u32(const uint32_t* keys_in, const uint32_t* vals_in, uint32_t* keys_out, uint32_t* vals_out, size_t n,
                   int end_bit, void* temp, bool profile, cudaStream_t stream)
{
    return sort_pairs_impl<uint32_t>(keys_in, vals_in, keys_out, vals_out, n, end_bit, temp, profile, 0, stream);
}

// have_hist == false: the control region is already zero (the caller's memset) but nobody has built the
// histograms: run the histogram + plan kernels here
int sort_pairs_u32_pre(const uint32_t* keys_in, const uint32_t* vals_in, uint32_t* keys_out, uint32_t* vals_out, size_t n,
                       int end_bit, void* temp, bool profile, bool have_hist, cudaStream_t stream, const uint32_t* n_dev)
{
    return sort_pairs_impl<uint32_t>(keys_in, vals_in, keys_out, vals_out, n, end_bit, temp, profile, have_hist ? 1 : 2, stream, n_dev);
}

size_t sort_zero_bytes(size_t n, size_t key_bytes, int end_bit)
{
    return SortTempLayout::make(n, key_bytes).zero_bytes(n, (end_bit + 7) / 8);
}

int sort_pre_handle(void* temp, size_t n, size_t key_bytes, int end_bit, SortPre* out)
{
    if (end_bit < 1 || end_bit > (int)(8 * key_bytes)) { set_error("sort: end_bit %d out of range", end_bit); return 1; }
    if (n >= (1ull << 30)) { set_error("sort: n=%zu exceeds 2^30", n); return 3; }
    SortTempLayout L = SortTempLayout::make(n, key_bytes);
    unsigned char* t = static_cast<unsigned char*>(temp);
    out->hist = reinterpret_cast<uint32_t*>(t + L.hist);
    out->ctl = reinterpret_cast<SortCtl*>(t + L.ctl);
    out->n = (uint32_t)n;
    out->n_dev = nullptr;
    out->npass = (end_bit + 7) / 8;
    out->end_bit = end_bit;
    return 0;
}

int sort_pre_begin(void* temp, size_t n, size_t key_bytes, int end_bit, SortPre* out, cudaStream_t stream)
{
    int rc = sort_pre_handle(temp, n, key_bytes, end_bit, out);
    if (rc) return rc;
    DMR_CUDA(cudaMemsetAsync(temp, 0, sort_zero_bytes(n, key_bytes, end_bit), stream));
    return 0;
}

}  // namespace dmr
