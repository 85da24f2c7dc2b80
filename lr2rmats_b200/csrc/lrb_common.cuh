// lrb_common.cuh -- shared device helpers for the lr2rmats_b200 kernels (sm_100a).
//
//  * single-pass chained scan ("decoupled look-back") over tiles handed out by a ticket counter, used wherever a kernel
//    must place variable-length per-read output compactly in read order while reading its input exactly once;
//  * warp / sub-warp (power-of-two lane group) reductions and scans on shuffles;
//  * cache-hinted 128-bit streaming loads / stores.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace lrbk {

#define LRB_DEVINL __device__ __forceinline__

static constexpr unsigned FULL = 0xffffffffu;

LRB_DEVINL int lane_id() { return threadIdx.x & 31; }
LRB_DEVINL int warp_id() { return threadIdx.x >> 5; }

// ---------------------------------------------------------------------------------------------- look-back scan
// tile state word: [63:62] status (0 invalid, 1 tile aggregate, 2 inclusive prefix), [61:0] value
static constexpr uint64_t LB_MASK = (1ull << 62) - 1;
static constexpr uint64_t LB_AGG = 1ull << 62, LB_INC = 2ull << 62;

struct OpAdd { LRB_DEVINL uint64_t operator()(uint64_t a, uint64_t b) const { return (a + b) & LB_MASK; } static constexpr uint64_t identity = 0; };
struct OpMax { LRB_DEVINL uint64_t operator()(uint64_t a, uint64_t b) const { return a > b ? a : b; } static constexpr uint64_t identity = 0; };
// two 31-bit counters packed as hi:lo (rows : exons); plain add works while neither half overflows 31 bits
static constexpr int PAIR_SHIFT = 31;
LRB_DEVINL uint64_t pack_pair(uint32_t hi, uint32_t lo) { return ((uint64_t)hi << PAIR_SHIFT) | lo; }
LRB_DEVINL uint32_t pair_hi(uint64_t v) { return (uint32_t)(v >> PAIR_SHIFT); }
LRB_DEVINL uint32_t pair_lo(uint64_t v) { return (uint32_t)(v & ((1ull << PAIR_SHIFT) - 1)); }

LRB_DEVINL uint64_t ld_volatile_u64(const uint64_t *p) { uint64_t v; asm volatile("ld.volatile.global.u64 %0, [%1];" : "=l"(v) : "l"(p)); return v; }
LRB_DEVINL void st_volatile_u64(uint64_t *p, uint64_t v) { asm volatile("st.volatile.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory"); }

// Called by ALL 32 lanes of one warp of the block.  `state` has one word per tile (zeroed before launch).
// Returns the exclusive prefix of tile `tile` under Op and publishes the inclusive one.
template <class Op>
LRB_DEVINL uint64_t lookback_exclusive(uint64_t *state, int tile, uint64_t aggregate, Op op)
{
    const int lane = lane_id();
    if (tile == 0) {
        if (lane == 0) { __threadfence(); st_volatile_u64(state, LB_INC | aggregate); }
        return Op::identity;
    }
    if (lane == 0) { __threadfence(); st_volatile_u64(state + tile, LB_AGG | aggregate); }
    uint64_t excl = Op::identity;
    int base = tile - 1;                       // nearest predecessor handled by lane 0
    for (;;) {
        int idx = base - lane;
        uint64_t w = LB_INC;                   // tiles before 0: identity, "inclusive"
        if (idx >= 0) { do { w = ld_volatile_u64(state + idx); } while ((w >> 62) == 0); }
        unsigned inc = __ballot_sync(FULL, (w >> 62) == 2);
        int stop = inc ? (__ffs(inc) - 1) : 32;         // first lane holding an inclusive prefix
        uint64_t v = (lane <= stop && idx >= 0) ? (w & LB_MASK) : Op::identity;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v = op(v, __shfl_xor_sync(FULL, v, o));
        excl = op(v, excl);
        if (inc) break;
        base -= 32;
    }
    if (lane == 0) { __threadfence(); st_volatile_u64(state + tile, LB_INC | op(excl, aggregate)); }
    return excl;
}

// ------------------------------------------------------------------------------------------------- block scans
// exclusive sum of one uint32 per thread across the block (blockDim.x multiple of 32, <= 1024); returns the
// exclusive prefix, total in *total (valid in every thread).  `sm` needs 33 words.
LRB_DEVINL uint32_t block_excl_sum(uint32_t v, uint32_t *sm, uint32_t *total)
{
    const int lane = lane_id(), w = warp_id(), nw = blockDim.x >> 5;
    uint32_t inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { uint32_t t = __shfl_up_sync(FULL, inc, o); if (lane >= o) inc += t; }
    if (lane == 31) sm[w] = inc;
    __syncthreads();
    if (w == 0) {
        uint32_t x = lane < nw ? sm[lane] : 0, xi = x;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { uint32_t t = __shfl_up_sync(FULL, xi, o); if (lane >= o) xi += t; }
        sm[lane] = xi - x;
        if (lane == 31) sm[32] = xi;
    }
    __syncthreads();
    uint32_t r = sm[w] + inc - v;
    *total = sm[32];
    __syncthreads();
    return r;
}

// ---------------------------------------------------------------------------------------------- lane groups
template <int G> LRB_DEVINL constexpr unsigned lane_bits() { return G >= 32 ? 0xffffffffu : ((1u << (G & 31)) - 1u); }
template <int G> LRB_DEVINL unsigned group_mask() { return G == 32 ? FULL : (lane_bits<G>() << ((lane_id() / G) * G)); }
// the shuffles name only the group's own lanes, so groups sharing a warp may diverge from each other
template <int G> LRB_DEVINL int group_sum(unsigned m, int v)
{
#pragma unroll
    for (int o = G / 2; o > 0; o >>= 1) v += __shfl_xor_sync(m, v, o);
    return v;
}
template <int G> LRB_DEVINL int group_or(unsigned m, int v)
{
#pragma unroll
    for (int o = G / 2; o > 0; o >>= 1) v |= __shfl_xor_sync(m, v, o);
    return v;
}

// first index in [lo, hi) with a[idx] > key (a non-decreasing)
template <class T> LRB_DEVINL int64_t upper_bound_dev(const T *a, int64_t lo, int64_t hi, T key)
{
    while (lo < hi) { int64_t mid = (lo + hi) >> 1; if (a[mid] > key) hi = mid; else lo = mid + 1; }
    return lo;
}
// first index in [lo, hi) with a[idx] >= key
template <class T> LRB_DEVINL int64_t lower_bound_dev(const T *a, int64_t lo, int64_t hi, T key)
{
    while (lo < hi) { int64_t mid = (lo + hi) >> 1; if (a[mid] < key) lo = mid + 1; else hi = mid; }
    return lo;
}

// cooperative (G+1)-ary searches: the G lanes of a group probe G pivots per step (one load each, in parallel), so a
// search over n keys costs ~log_{G+1}(n) dependent loads instead of log_2(n).  `a` non-decreasing; all lanes of the
// group must call with the same arguments and receive the same result.  A group of one lane runs the plain binary search.
template <int G, class T> LRB_DEVINL int64_t group_upper_bound(unsigned m, int gl, const T *a, int64_t lo, int64_t hi, T key)
{
    if constexpr (G == 1) return upper_bound_dev(a, lo, hi, key);
    const int sh = (lane_id() / G) * G;
    while (hi - lo > G) {
        const int64_t span = hi - lo;
        const int64_t p = lo + (span * (gl + 1)) / (G + 1);            // lo <= p < hi, strictly increasing in gl
        const unsigned b = (__ballot_sync(m, a[p] > key) >> sh) & lane_bits<G>();
        if (b) {
            const int f = __ffs(b) - 1;                                  // first pivot above the key
            const int64_t pf = lo + (span * (f + 1)) / (G + 1);
            const int64_t pl = f ? lo + (span * f) / (G + 1) + 1 : lo;
            lo = pl; hi = pf;
        } else lo = lo + (span * G) / (G + 1) + 1;
    }
    const int64_t q = lo + gl;
    const unsigned b = (__ballot_sync(m, q < hi && a[q] > key) >> sh) & lane_bits<G>();
    return b ? lo + (__ffs(b) - 1) : hi;
}
template <int G, class T> LRB_DEVINL int64_t group_lower_bound(unsigned m, int gl, const T *a, int64_t lo, int64_t hi, T key)
{
    if constexpr (G == 1) return lower_bound_dev(a, lo, hi, key);
    const int sh = (lane_id() / G) * G;
    while (hi - lo > G) {
        const int64_t span = hi - lo;
        const int64_t p = lo + (span * (gl + 1)) / (G + 1);
        const unsigned b = (__ballot_sync(m, a[p] >= key) >> sh) & lane_bits<G>();
        if (b) {
            const int f = __ffs(b) - 1;
            const int64_t pf = lo + (span * (f + 1)) / (G + 1);
            const int64_t pl = f ? lo + (span * f) / (G + 1) + 1 : lo;
            lo = pl; hi = pf;
        } else lo = lo + (span * G) / (G + 1) + 1;
    }
    const int64_t q = lo + gl;
    const unsigned b = (__ballot_sync(m, q < hi && a[q] >= key) >> sh) & lane_bits<G>();
    return b ? lo + (__ffs(b) - 1) : hi;
}

// --------------------------------------------------------------------------------------------- memory helpers
LRB_DEVINL uint4 ldg_stream_u4(const uint4 *p) { uint4 r; asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p)); return r; }
LRB_DEVINL uint32_t ldg_stream_u32(const uint32_t *p) { uint32_t r; asm volatile("ld.global.nc.L1::no_allocate.u32 %0, [%1];" : "=r"(r) : "l"(p)); return r; }

LRB_DEVINL int iabs_dev(int x) { return x < 0 ? -x : x; }

}  // namespace lrbk
