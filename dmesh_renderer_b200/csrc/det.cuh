// det.cuh -- fixed-point accumulation for the deterministic (run-to-run reproducible) backward passes.
#pragma once
#include "common.cuh"

namespace dmr {

// Deterministic mode (SURVEY.md 8f-3)
// ----------------------------------
// Everything up to the gradient accumulation is already run-to-run reproducible (stable sorts, fixed per-pixel
// compositing order); only the ORDER in which the groups' partial sums reach a (view, face) record, and the faces'
// contributions reach a vertex, varies -- and fp32 addition is not associative.  The deterministic variant
// accumulates the same partial sums as FIXED-POINT integers (integer addition is associative, so any arrival order
// gives the same bits), added with red.global.add.u64.
// All gradients are linear in the cotangent, so the binary point is placed relative to g = max |dL_dout| (found by a
// max-reduction, itself order-independent): with 2^(e-1) <= g < 2^e, a term x is accumulated in units of 2^(e-k),
//     colour / opacity / intensity / depth terms:  k = 48   (resolution 2^(e-48) <= 7.1e-15 g)
//     vertex-position terms (carry t and 1/det):   k = 40   (resolution 2^(e-40) <= 1.8e-12 g)
// An accumulator is TWO 64-bit words.  A term, in units of 2^32 of the low word (det_scales), is split exactly into
// its integer part h, added to the high word, and its fraction rounded to 32 bits, |l| <= 2^32, added to the low
// word; zero parts are not added.  The low word cannot wrap for fewer than 2^31 terms per accumulator; the high word
// holds the sum exactly while |sum| < 2^(95-k+e), i.e. beyond 2^47 g for values and 2^55 g for positions.  A
// single term of 2^62 high units or more (never below 2^46 g / 2^54 g), and a NaN term, raises the overflow word
// instead, and the convert kernels then POISON every fixed-point gradient of the call with NaN.  Only a sum of
// several terms each below that cap can pass 2^(95-k+e) unflagged: at least 2^47 g of gradient in one accumulator.
// (A single word with 38 bits below g would wrap from 2^25 g on, which a face over an eighth of a 1024^2 screen in a
// 64-view call under an L1 loss reaches.)
// The high words mirror the low ones at a fixed element offset `hi` (the layouts in tri.cuh / tet.cuh), so an
// accumulator is addressed by its low word alone.
#define DMR_DET_VALUE_BITS 48
#define DMR_DET_GEOM_BITS 40
#define DMR_DET_MIN_EXP (DMR_DET_VALUE_BITS - 32 - 127)    // scales stay finite floats: 2^(k-32-e) <= 2^127
// sv, sg: scales from a gradient value to HIGH-word units, 2^(k-32-e); 0 when all cotangents are zero (all gradients
// are zero) or g is not finite.  Below g = 2^(DMR_DET_MIN_EXP-1) = 2^-112 ~ 1.9e-34 the binary point stops following g.
__device__ __forceinline__ void det_scales(uint32_t gmax_bits, float& sv, float& sg)
{
    const float g = __uint_as_float(gmax_bits);
    sv = sg = 0.0f;
    if (!(g > 0.0f) || !(g <= 3.40282347e38f)) return;       // zero, inf or NaN cotangents
    int e;
    frexpf(g, &e);
    e = max(e, DMR_DET_MIN_EXP);
    sv = ldexpf(1.0f, DMR_DET_VALUE_BITS - 32 - e);
    sg = ldexpf(1.0f, DMR_DET_GEOM_BITS - 32 - e);
}
// gmax[0]: bits of g; gmax[1]: overflow word (det_add).  Non-finite cotangents (inf / NaN bit patterns order above
// every finite float) or a term beyond the range: the fixed-point format has no representation for them, so the
// convert kernels POISON the gradients with NaN -- as the fp32-atomic path and the reference would propagate a
// non-finite cotangent -- instead of returning zeros or a wrapped sum, which would look like a clean step.
__device__ __forceinline__ bool det_poisoned(const uint32_t* gmax) { return gmax[0] >= 0x7f800000u || gmax[1] != 0u; }
__device__ __forceinline__ void det_add(long long* dst, float v, float scale, ptrdiff_t hi, const uint32_t* gmax)
{
    const float x = v * scale;                                   // high-word units (a power-of-two scale: exact)
    if (!(fabsf(x) < 0x1p62f)) {                                 // beyond the range, or NaN
        *const_cast<uint32_t*>(gmax + 1) = 1u;
        return;
    }
    const float h = truncf(x);
    const long long qh = (long long)h;                           // exact: |h| < 2^62 is an integer
    const long long ql = __float2ll_rn((x - h) * 0x1p32f);      // the fraction x - h is exact, |ql| <= 2^32
    if (ql != 0) atomicAdd(reinterpret_cast<unsigned long long*>(dst), static_cast<unsigned long long>(ql));
    if (qh != 0) atomicAdd(reinterpret_cast<unsigned long long*>(dst + hi), static_cast<unsigned long long>(qh));
}
// Value of the accumulator whose low word is *lo, in units of 1 / scale (inv = 1 / scale).
__device__ __forceinline__ double det_value(const long long* lo, ptrdiff_t hi, double inv)
{
    return ((double)lo[hi] + (double)lo[0] * 0x1p-32) * inv;
}
__device__ __forceinline__ bool det_nonzero(const long long* lo, ptrdiff_t hi) { return (lo[0] | lo[hi]) != 0; }

// g = max |dL_dout| over both cotangent images, as float bits, into *gmax (zeroed by the caller).
int det_gmax(const float* a, size_t na, const float* b, size_t nb, uint32_t* gmax, cudaStream_t stream);

}  // namespace dmr
