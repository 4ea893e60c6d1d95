// gpu_build.cu -- device-side construction of the flattened ball tree; see gpu_build.hpp.
// Compiled with -fmad=false like the rest of the library: centroid sums and radius folds must round exactly as the host
// builder's (and the reference's) separate multiply and add.
#include "gpu_build.hpp"

#include <float.h>

#include <algorithm>
#include <cstring>

namespace petal {
namespace gb {

#define GB_CU(x)                                                           \
    do {                                                                   \
        cudaError_t e_ = (x);                                              \
        if (e_ != cudaSuccess) {                                           \
            err = std::string(#x) + ": " + cudaGetErrorString(e_);         \
            return (int)e_;                                                \
        }                                                                  \
    } while (0)

constexpr int BT = 256;     // threads per block of every builder kernel
constexpr uint32_t TILE_ROWS = 128;  // rows per tile of the tensor path's point image (tc::BN)
constexpr int ROWS = 1024;  // consecutive positions of ONE segment handled by a block (blocks never straddle segments)

template <typename A> struct KeyT;
template <> struct KeyT<float>  { using U = uint32_t;           static constexpr int VB = 4; };
template <> struct KeyT<double> { using U = unsigned long long; static constexpr int VB = 8; };

// order-preserving map float -> unsigned; -0 is folded into +0 first so that equal values get equal keys (the host
// comparison `va < vb || (va == vb && a < b)` treats them as equal)
__device__ __forceinline__ uint32_t ord_key(float v) {
    const uint32_t u = __float_as_uint(v + 0.0f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ unsigned long long ord_key(double v) {
    const unsigned long long u = (unsigned long long)__double_as_longlong(v + 0.0);
    return (u >> 63) ? ~u : (u | 0x8000000000000000ull);
}
__device__ __forceinline__ float ord_val(uint32_t k) { return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k); }
__device__ __forceinline__ double ord_val(unsigned long long k) {
    return __longlong_as_double((long long)((k >> 63) ? (k & 0x7fffffffffffffffull) : ~k));
}

// block b of a level -> (segment, first position, count): cps blocks per segment, ROWS positions each
struct Span { uint32_t seg, lo, cnt, seg_lo, seg_hi; };
// (ball trees: seg_hi = seg_lo + 1, the boundaries of a level are contiguous; vantage-point trees keep separate arrays --
// the vantage point of a node sits between its children's ranges)
__device__ __forceinline__ Span block_span(const uint32_t* __restrict__ seg_lo, const uint32_t* __restrict__ seg_hi, uint32_t cps) {
    Span s;
    s.seg = blockIdx.x / cps;
    const uint32_t chunk = blockIdx.x % cps;
    s.seg_lo = seg_lo[s.seg]; s.seg_hi = seg_hi[s.seg];
    const uint64_t lo = (uint64_t)s.seg_lo + (uint64_t)chunk * ROWS;
    s.lo = (uint32_t)min(lo, (uint64_t)s.seg_hi);
    s.cnt = min((uint32_t)ROWS, s.seg_hi - s.lo);
    return s;
}

// ---- 1. per-segment, per-column min / max (max_spread_column, src/ball_tree.rs:577-603) -----------------------------
template <typename A>
__global__ void __launch_bounds__(BT) minmax_kernel(const A* __restrict__ raw, uint64_t stride, uint32_t d, const uint32_t* __restrict__ idx,
                                                    const uint32_t* __restrict__ seg_l, const uint32_t* __restrict__ seg_h, uint32_t cps,
                                                    typename KeyT<A>::U* __restrict__ mn, typename KeyT<A>::U* __restrict__ mx) {
    using U = typename KeyT<A>::U;
    __shared__ U s_mn[BT], s_mx[BT];
    const Span sp = block_span(seg_l, seg_h, cps);
    if (sp.cnt == 0) return;
    uint32_t dp = 1;
    while (dp < d && dp < BT) dp <<= 1;            // threads per row (power of two <= 256)
    const uint32_t rpar = BT / dp;                 // rows in flight
    const uint32_t c0 = threadIdx.x % dp, rs = threadIdx.x / dp;
    for (uint32_t cb = 0; cb < d; cb += dp) {
        const uint32_t c = cb + c0;
        U lo = ~(U)0, hi = 0;
        if (c < d) {
            for (uint32_t r = rs; r < sp.cnt; r += rpar) {
                const U k = ord_key(raw[(uint64_t)idx[sp.lo + r] * stride + c]);
                lo = min(lo, k); hi = max(hi, k);
            }
        }
        s_mn[threadIdx.x] = lo; s_mx[threadIdx.x] = hi;
        __syncthreads();
        if (rs == 0 && c < d) {
            for (uint32_t k = 1; k < rpar; ++k) { lo = min(lo, s_mn[c0 + k * dp]); hi = max(hi, s_mx[c0 + k * dp]); }
            atomicMin(&mn[(uint64_t)sp.seg * d + c], lo);
            atomicMax(&mx[(uint64_t)sp.seg * d + c], hi);
        }
        __syncthreads();
    }
}

// first column with the strictly greatest spread (src/ball_tree.rs:604-612)
template <typename A>
__global__ void choose_kernel(const typename KeyT<A>::U* __restrict__ mn, const typename KeyT<A>::U* __restrict__ mx, uint32_t d,
                              uint32_t n_seg, const uint32_t* __restrict__ seg_l, const uint32_t* __restrict__ seg_h, uint32_t* __restrict__ col) {
    const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n_seg) return;
    uint32_t best_c = 0;
    if (seg_h[s] - seg_l[s] >= 2) {
        A best = ord_val(mx[(uint64_t)s * d]) - ord_val(mn[(uint64_t)s * d]);
        for (uint32_t j = 1; j < d; ++j) {
            const A sp = ord_val(mx[(uint64_t)s * d + j]) - ord_val(mn[(uint64_t)s * d + j]);
            if (sp > best) { best = sp; best_c = j; }
        }
    }
    col[s] = best_c;
}

// ---- 1b. the TWO-MEANS split rule (rule 1; not the reference's): the split direction of a segment is the line through
// the two centroids of a 2-means clustering of a sample of its points, the key of a point its projection on that line.
// The median cut, the stable partition and everything after stay as they are, so the result is a ball tree of the same
// shape with correct centroids and radii -- every query path is exact on it -- whose buckets follow clusters instead of
// cutting through them along coordinate axes (what the tile bounds of the pruned tensor scan need, tc_prune.cuh).
// One block per segment: up to `m_max` evenly spaced points of the segment in shared memory, two far-apart seeds (the
// point farthest from the first sample, then the point farthest from that one), four Lloyd iterations, all reductions in
// a fixed order (the layout is reproducible run to run).
template <typename A>
__global__ void __launch_bounds__(BT) two_means_dir_kernel(const A* __restrict__ raw, uint64_t stride, uint32_t d, const uint32_t* __restrict__ idx,
                                                           const uint32_t* __restrict__ seg_l, const uint32_t* __restrict__ seg_h, uint32_t m_max,
                                                           A* __restrict__ wdir) {
    extern __shared__ __align__(16) unsigned char dir_smem[];
    const uint32_t ds = d | 1u;                                // odd row stride: lane i reads row i without bank conflicts
    float* S = reinterpret_cast<float*>(dir_smem);             // [m_max][ds]
    float* c1 = S + (size_t)m_max * ds;                        // [d]
    float* c2 = c1 + d;                                        // [d]
    __shared__ float s_val[BT];
    __shared__ uint32_t s_idx[BT];
    __shared__ uint32_t s_grp[BT];
    __shared__ uint32_t s_n1;
    const uint32_t seg = blockIdx.x;
    const uint32_t lo = seg_l[seg], len = seg_h[seg] - lo;
    A* w = wdir + (uint64_t)seg * d;
    if (len < 2) {   // nothing to split
        for (uint32_t j = threadIdx.x; j < d; j += BT) w[j] = A(0);
        return;
    }
    const uint32_t m = min(len, m_max);
    for (uint32_t e = threadIdx.x; e < m * d; e += BT) {
        const uint32_t i = e / d, j = e % d;
        const uint32_t pos = (uint32_t)(((uint64_t)i * len) / m);
        S[(size_t)i * ds + j] = (float)raw[(uint64_t)idx[lo + pos] * stride + j];
    }
    __syncthreads();
    // sample farthest from row `from` (ties: the lower sample), by a fixed-order tree reduction
    auto farthest = [&](const float* from) -> uint32_t {
        float v = -1.f;
        if (threadIdx.x < m) {
            v = 0.f;
            const float* r = S + (size_t)threadIdx.x * ds;
            for (uint32_t j = 0; j < d; ++j) { const float t = r[j] - from[j]; v += t * t; }
        }
        s_val[threadIdx.x] = v; s_idx[threadIdx.x] = threadIdx.x;
        __syncthreads();
        for (uint32_t o = BT / 2; o; o >>= 1) {
            if (threadIdx.x < o) {
                const float a = s_val[threadIdx.x], b = s_val[threadIdx.x + o];
                if (b > a) { s_val[threadIdx.x] = b; s_idx[threadIdx.x] = s_idx[threadIdx.x + o]; }
            }
            __syncthreads();
        }
        const uint32_t best = s_idx[0];
        __syncthreads();
        return best;
    };
    const uint32_t ib = farthest(S);
    for (uint32_t j = threadIdx.x; j < d; j += BT) c1[j] = S[(size_t)ib * ds + j];
    __syncthreads();
    const uint32_t ic = farthest(c1);
    for (uint32_t j = threadIdx.x; j < d; j += BT) c2[j] = S[(size_t)ic * ds + j];
    __syncthreads();
    for (int it = 0; it < 4; ++it) {
        if (threadIdx.x == 0) s_n1 = 0;
        __syncthreads();
        uint32_t g = 2;   // 0: nearer c1, 1: nearer c2, 2: no such sample
        if (threadIdx.x < m) {
            const float* r = S + (size_t)threadIdx.x * ds;
            float d1 = 0.f, d2 = 0.f;
            for (uint32_t j = 0; j < d; ++j) {
                const float t1 = r[j] - c1[j], t2 = r[j] - c2[j];
                d1 += t1 * t1; d2 += t2 * t2;
            }
            g = d1 <= d2 ? 0u : 1u;
            if (g == 0) atomicAdd(&s_n1, 1u);   // an integer count: order-independent
        }
        s_grp[threadIdx.x] = g;
        __syncthreads();
        const uint32_t n1 = s_n1, n2 = m - n1;
        if (n1 == 0 || n2 == 0) break;          // block-uniform: one side is empty (identical samples), keep the centroids
        for (uint32_t j = threadIdx.x; j < d; j += BT) {
            float a1 = 0.f, a2 = 0.f;
            for (uint32_t i = 0; i < m; ++i) {
                const float v = S[(size_t)i * ds + j];
                if (s_grp[i] == 0) a1 += v; else a2 += v;
            }
            c1[j] = a1 / (float)n1; c2[j] = a2 / (float)n2;
        }
        __syncthreads();
    }
    __syncthreads();
    for (uint32_t j = threadIdx.x; j < d; j += BT) w[j] = (A)(c2[j] - c1[j]);
}

// key of a point = its projection on the direction of its segment: a warp per row, the lanes over the columns, partial
// sums combined in a fixed butterfly order
template <typename A>
__global__ void __launch_bounds__(BT) proj_keys_kernel(const A* __restrict__ raw, uint64_t stride, uint32_t d, const uint32_t* __restrict__ idx,
                                                       const uint32_t* __restrict__ seg_l, const uint32_t* __restrict__ seg_h, uint32_t cps,
                                                       const A* __restrict__ wdir, typename KeyT<A>::U* __restrict__ kv) {
    const Span sp = block_span(seg_l, seg_h, cps);
    if (sp.cnt == 0) return;
    const A* w = wdir + (uint64_t)sp.seg * d;
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (uint32_t r = warp; r < sp.cnt; r += BT / 32) {
        const A* row = raw + (uint64_t)idx[sp.lo + r] * stride;
        A acc = A(0);
        for (uint32_t j = lane; j < d; j += 32) acc += row[j] * w[j];
        for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        if (lane == 0) kv[sp.lo + r] = ord_key(acc);
    }
}

// ---- 2. median of each segment on the (value of the split column, original index) key: MSB-first radix select -------
template <typename A>
__global__ void __launch_bounds__(BT) keys_kernel(const A* __restrict__ raw, uint64_t stride, const uint32_t* __restrict__ idx,
                                                  const uint32_t* __restrict__ seg_l, const uint32_t* __restrict__ seg_h, uint32_t cps, const uint32_t* __restrict__ col,
                                                  typename KeyT<A>::U* __restrict__ kv) {
    const Span sp = block_span(seg_l, seg_h, cps);
    const uint32_t c = col[sp.seg];
    for (uint32_t r = threadIdx.x; r < sp.cnt; r += BT) kv[sp.lo + r] = ord_key(raw[(uint64_t)idx[sp.lo + r] * stride + c]);
}

template <typename U> struct SelState { U pv; uint32_t pi; uint32_t m; };

// rank of the element a select is after, by `mode`: 0 = len / 2 (ball: mid - start, src/ball_tree.rs:535-537),
// 1 = len - 1 (the maximum: a vantage point is the LAST element of its sorted slice, src/vantage_point_tree.rs:169-170),
// 2 = (len - 1) / 2 (far[0] of the slice without its vantage point, :180-182)
__device__ __forceinline__ uint32_t select_rank(uint32_t len, int mode) {
    return mode == 0 ? len / 2 : (mode == 1 ? len - 1 : (len - 1) / 2);
}
template <typename U>
__global__ void init_state_kernel(const uint32_t* __restrict__ seg_l, const uint32_t* __restrict__ seg_h, uint32_t n_seg, int mode,
                                  SelState<U>* __restrict__ st, const uint32_t* __restrict__ seg_next = nullptr) {
    const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n_seg) return;
    const uint32_t len = seg_h[s] - seg_l[s];
    // seg_next: the split position is whatever the shape says (tile-aligned shapes), boundary 2s+1 of the next level
    st[s].pv = 0; st[s].pi = 0; st[s].m = len ? (seg_next ? seg_next[2 * s + 1] - seg_l[s] : select_rank(len, mode)) : 0;
}

template <typename U, int VB>
__device__ __forceinline__ bool sel_match(U kv, uint32_t id, const SelState<U>& s, int pass) {
    if (pass == 0) return true;
    if (pass <= VB) { const int sh = 8 * (VB - pass); return (kv >> sh) == (s.pv >> sh); }
    const int sh = 8 * (4 - (pass - VB));
    return kv == s.pv && (id >> sh) == (s.pi >> sh);
}
template <typename U, int VB>
__device__ __forceinline__ uint32_t sel_digit(U kv, uint32_t id, int pass) {
    return pass < VB ? (uint32_t)(kv >> (8 * (VB - 1 - pass))) & 255u : (id >> (8 * (3 - (pass - VB)))) & 255u;
}
template <typename U, int VB>
__device__ __forceinline__ void sel_extend(SelState<U>& s, uint32_t dg, uint32_t before, int pass) {
    if (pass < VB) s.pv |= (U)dg << (8 * (VB - 1 - pass)); else s.pi |= dg << (8 * (3 - (pass - VB)));
    s.m -= before;
}

// large segments: one pass = histogram over many blocks + a pick kernel
template <typename A>
__global__ void __launch_bounds__(BT) hist_kernel(const typename KeyT<A>::U* __restrict__ kv, const uint32_t* __restrict__ idx,
                                                  const uint32_t* __restrict__ seg_l, const uint32_t* __restrict__ seg_h, uint32_t cps,
                                                  const SelState<typename KeyT<A>::U>* __restrict__ st, int pass, uint32_t* __restrict__ hist) {
    using U = typename KeyT<A>::U;
    __shared__ uint32_t sh[256];
    const Span sp = block_span(seg_l, seg_h, cps);
    if (sp.cnt == 0) return;
    sh[threadIdx.x] = 0;
    __syncthreads();
    const SelState<U> s = st[sp.seg];
    for (uint32_t r = threadIdx.x; r < sp.cnt; r += BT) {
        const U k = kv[sp.lo + r];
        const uint32_t id = idx[sp.lo + r];
        if (sel_match<U, KeyT<A>::VB>(k, id, s, pass)) atomicAdd(&sh[sel_digit<U, KeyT<A>::VB>(k, id, pass)], 1u);
    }
    __syncthreads();
    if (sh[threadIdx.x]) atomicAdd(&hist[(uint64_t)sp.seg * 256 + threadIdx.x], sh[threadIdx.x]);
}
template <typename U, int VB>
__global__ void pick_kernel(uint32_t* __restrict__ hist, SelState<U>* __restrict__ st, const uint32_t* __restrict__ seg_l,
                            const uint32_t* __restrict__ seg_h, uint32_t n_seg, int pass) {
    const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n_seg) return;
    uint32_t* h = hist + (uint64_t)s * 256;
    if (seg_h[s] > seg_l[s]) {
        SelState<U> x = st[s];
        uint32_t run = 0, dg = 0;
        for (; dg < 256; ++dg) {
            const uint32_t c = h[dg];
            if (run + c > x.m) break;
            run += c;
        }
        sel_extend<U, VB>(x, dg, run, pass);
        st[s] = x;
    }
    for (uint32_t dg = 0; dg < 256; ++dg) h[dg] = 0;
}
// small segments (at most SMALL_MAX points): one block per segment runs every pass on a shared-memory histogram
constexpr uint32_t SMALL_MAX = 4096;
template <typename A>
__global__ void __launch_bounds__(BT) select_small_kernel(const typename KeyT<A>::U* __restrict__ kv, const uint32_t* __restrict__ idx,
                                                          const uint32_t* __restrict__ seg_l, const uint32_t* __restrict__ seg_h, int mode,
                                                          SelState<typename KeyT<A>::U>* __restrict__ st, const uint32_t* __restrict__ seg_next = nullptr) {
    using U = typename KeyT<A>::U;
    constexpr int VB = KeyT<A>::VB;
    __shared__ uint32_t sh[256];
    __shared__ SelState<U> s;
    const uint32_t seg = blockIdx.x, lo = seg_l[seg], cnt = seg_h[seg] - lo;
    if (cnt == 0) return;
    if (threadIdx.x == 0) { s.pv = 0; s.pi = 0; s.m = seg_next ? seg_next[2 * seg + 1] - lo : select_rank(cnt, mode); }
    for (int pass = 0; pass < VB + 4; ++pass) {
        sh[threadIdx.x] = 0;
        __syncthreads();
        const SelState<U> cur = s;
        for (uint32_t r = threadIdx.x; r < cnt; r += BT) {
            const U k = kv[lo + r];
            const uint32_t id = idx[lo + r];
            if (sel_match<U, VB>(k, id, cur, pass)) atomicAdd(&sh[sel_digit<U, VB>(k, id, pass)], 1u);
        }
        __syncthreads();
        if (threadIdx.x < 32) {  // warp 0: lane l owns bins 8l .. 8l+7
            uint32_t c[8], tot = 0;
            for (int i = 0; i < 8; ++i) { c[i] = sh[threadIdx.x * 8 + i]; tot += c[i]; }
            uint32_t incl = tot;
            for (int o = 1; o < 32; o <<= 1) { const uint32_t v = __shfl_up_sync(0xffffffffu, incl, o); if ((int)threadIdx.x >= o) incl += v; }
            const unsigned hit = __ballot_sync(0xffffffffu, incl > cur.m);
            const int lane = __ffs(hit) - 1;  // cur.m < number of matching elements, so some lane qualifies
            if ((int)threadIdx.x == lane) {
                uint32_t run = incl - tot, dg = 0;
                for (; dg < 8; ++dg) { if (run + c[dg] > cur.m) break; run += c[dg]; }
                SelState<U> x = cur;
                sel_extend<U, VB>(x, threadIdx.x * 8 + dg, run, pass);
                s = x;
            }
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) st[seg] = s;
}

// the cut of every node of a level, for routing queries the way the points were split (home_bucket_planes_kernel):
// direction (zero padded to dpad) and the key of the pivot -- keys below it went to the left child
template <typename A>
__global__ void save_planes_kernel(const A* __restrict__ wdir, const SelState<typename KeyT<A>::U>* __restrict__ st, const uint32_t* __restrict__ seg_l,
                                   const uint32_t* __restrict__ seg_h, uint32_t n_seg, uint32_t first, uint32_t d, uint32_t dpad,
                                   A* __restrict__ plane_w, A* __restrict__ plane_t) {
    const uint32_t e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n_seg * dpad) return;
    const uint32_t s = e / dpad, j = e % dpad;
    const bool live = seg_h[s] - seg_l[s] >= 2;   // shorter segments were not split: everything "goes right" of -inf, harmlessly
    plane_w[(uint64_t)(first + s) * dpad + j] = live && j < d ? wdir[(uint64_t)s * d + j] : A(0);
    if (j == 0) plane_t[first + s] = live ? ord_val(st[s].pv) : A(0);
}

// ---- 3. stable partition around the pivot: keys below it go to the left child, order (ascending original index) kept --
template <typename U>
__device__ __forceinline__ bool goes_left(U k, uint32_t id, const SelState<U>& s) { return k < s.pv || (k == s.pv && id < s.pi); }

template <typename A>
__global__ void __launch_bounds__(BT) count_left_kernel(const typename KeyT<A>::U* __restrict__ kv, const uint32_t* __restrict__ idx,
                                                        const uint32_t* __restrict__ seg_l, const uint32_t* __restrict__ seg_h, uint32_t cps,
                                                        const SelState<typename KeyT<A>::U>* __restrict__ st, uint32_t* __restrict__ csum) {
    using U = typename KeyT<A>::U;
    __shared__ uint32_t wsum[BT / 32];
    const Span sp = block_span(seg_l, seg_h, cps);
    uint32_t c = 0;
    if (sp.cnt) {
        const SelState<U> s = st[sp.seg];
        for (uint32_t r = threadIdx.x; r < sp.cnt; r += BT) c += goes_left<U>(kv[sp.lo + r], idx[sp.lo + r], s) ? 1u : 0u;
    }
    c = __reduce_add_sync(0xffffffffu, c);
    if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) { uint32_t t = 0; for (int w = 0; w < BT / 32; ++w) t += wsum[w]; csum[blockIdx.x] = t; }
}
// exclusive scan of nb block counts, one block (nb <= a few hundred thousand)
__global__ void scan_blocks_kernel(const uint32_t* __restrict__ in, uint32_t* __restrict__ out, uint32_t nb) {
    __shared__ uint32_t sums[1024];
    const uint32_t tid = threadIdx.x, nt = blockDim.x;
    const uint32_t chunk = (nb + nt - 1) / nt;
    const uint32_t b = min(nb, tid * chunk), e = min(nb, b + chunk);
    uint32_t s = 0;
    for (uint32_t i = b; i < e; ++i) s += in[i];
    sums[tid] = s;
    __syncthreads();
    if (tid == 0) { uint32_t run = 0; for (uint32_t i = 0; i < nt; ++i) { const uint32_t v = sums[i]; sums[i] = run; run += v; } }
    __syncthreads();
    uint32_t run = sums[tid];
    for (uint32_t i = b; i < e; ++i) { const uint32_t v = in[i]; out[i] = run; run += v; }
}
template <typename A>
__global__ void __launch_bounds__(BT) scatter_kernel(const typename KeyT<A>::U* __restrict__ kv, const uint32_t* __restrict__ idx,
                                                     const uint32_t* __restrict__ seg_l, const uint32_t* __restrict__ seg_h, const uint32_t* __restrict__ seg_next, uint32_t cps,
                                                     const SelState<typename KeyT<A>::U>* __restrict__ st, const uint32_t* __restrict__ cex,
                                                     uint32_t* __restrict__ idx_out) {
    using U = typename KeyT<A>::U;
    __shared__ uint32_t wsum[BT / 32];
    const Span sp = block_span(seg_l, seg_h, cps);
    if (sp.cnt == 0) return;
    const SelState<U> s = st[sp.seg];
    const uint32_t mid = seg_next[2 * sp.seg + 1];
    const uint32_t left_before = cex[blockIdx.x] - cex[sp.seg * cps];     // left-goers of this segment in earlier blocks
    // thread t owns positions 4t .. 4t+3 of the block, so thread order is position order
    constexpr int PER = ROWS / BT;
    uint32_t ids[PER]; bool lf[PER];
    uint32_t mine = 0;
#pragma unroll
    for (int i = 0; i < PER; ++i) {
        const uint32_t r = threadIdx.x * PER + i;
        lf[i] = false; ids[i] = 0;
        if (r < sp.cnt) { ids[i] = idx[sp.lo + r]; lf[i] = goes_left<U>(kv[sp.lo + r], ids[i], s); mine += lf[i] ? 1u : 0u; }
    }
    uint32_t incl = mine;
    for (int o = 1; o < 32; o <<= 1) { const uint32_t v = __shfl_up_sync(0xffffffffu, incl, o); if ((int)(threadIdx.x & 31) >= o) incl += v; }
    if ((threadIdx.x & 31) == 31) wsum[threadIdx.x >> 5] = incl;
    __syncthreads();
    uint32_t wbase = 0;
    for (uint32_t w = 0; w < (threadIdx.x >> 5); ++w) wbase += wsum[w];
    uint32_t lrun = left_before + wbase + incl - mine;                      // left-goers of the segment before my first position
#pragma unroll
    for (int i = 0; i < PER; ++i) {
        const uint32_t r = threadIdx.x * PER + i;
        if (r >= sp.cnt) break;
        const uint32_t pos_in_seg = sp.lo + r - sp.seg_lo;
        const uint32_t dst = lf[i] ? sp.seg_lo + lrun : mid + (pos_in_seg - lrun);
        idx_out[dst] = ids[i];
        lrun += lf[i] ? 1u : 0u;
    }
}

// ---- 4. flatten + Node::init for every node (src/ball_tree.rs:445-461) ----------------------------------------------
__global__ void iota_kernel(uint32_t* __restrict__ idx, uint64_t n) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) idx[i] = (uint32_t)i;
}
template <typename A>
__global__ void gather_rows_kernel(const A* __restrict__ raw, uint64_t stride, uint32_t d, uint32_t dpad, const uint32_t* __restrict__ idx,
                                   uint64_t n, A* __restrict__ pts, uint32_t* __restrict__ ids) {
    const uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n * dpad) return;
    const uint64_t i = e / dpad;
    const uint32_t j = (uint32_t)(e % dpad);
    const uint32_t src = idx[i];
    pts[e] = j < d ? raw[(uint64_t)src * stride + j] : A(0);
    if (j == 0) ids[i] = src;
}
// bucket sums: sequential over the bucket's rows in stored order, one thread per column (the host's `acc[j] += r[j]`)
template <typename A>
__global__ void bucket_sum_kernel(const A* __restrict__ pts, uint32_t d, uint32_t dpad, const uint32_t* __restrict__ bucket_seg,
                                  uint32_t n_internal, A* __restrict__ sums) {
    const uint32_t b = blockIdx.x;
    const uint32_t lo = bucket_seg[b], hi = bucket_seg[b + 1];
    for (uint32_t j = threadIdx.x; j < d; j += blockDim.x) {
        A acc = A(0);
        for (uint32_t i = lo; i < hi; ++i) acc = acc + pts[(uint64_t)i * dpad + j];
        sums[(uint64_t)(n_internal + b) * dpad + j] = acc;
    }
}
// one level of internal nodes: sum = left child + right child
template <typename A>
__global__ void node_sum_kernel(A* __restrict__ sums, uint32_t first, uint32_t count, uint32_t d, uint32_t dpad) {
    const uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= (uint64_t)count * d) return;
    const uint32_t node = first + (uint32_t)(e / d), j = (uint32_t)(e % d);
    sums[(uint64_t)node * dpad + j] = sums[(uint64_t)(2 * node + 1) * dpad + j] + sums[(uint64_t)(2 * node + 2) * dpad + j];
}
__device__ __forceinline__ float  xdiv(float a, float b)   { return __fdiv_rn(a, b); }
__device__ __forceinline__ double xdiv(double a, double b) { return __ddiv_rn(a, b); }
template <typename A>
__global__ void centroid_kernel(A* __restrict__ centers, A* __restrict__ radii, const uint32_t* __restrict__ cnt, uint32_t n_nodes, uint32_t d,
                                uint32_t dpad) {
    const uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= (uint64_t)n_nodes * dpad) return;
    const uint32_t node = (uint32_t)(e / dpad), j = (uint32_t)(e % dpad);
    const uint32_t c = cnt[node];
    centers[e] = (c && j < d) ? xdiv(centers[e], (A)c) : A(0);
    if (j == 0) radii[node] = A(0);
}
__device__ __forceinline__ void atomic_max_nonneg(float* p, float v) { atomicMax(reinterpret_cast<unsigned int*>(p), __float_as_uint(v)); }
__device__ __forceinline__ void atomic_max_nonneg(double* p, double v) {
    atomicMax(reinterpret_cast<unsigned long long*>(p), (unsigned long long)__double_as_longlong(v));
}
__device__ __forceinline__ float  xsqrt_rn(float a)  { return __fsqrt_rn(a); }
__device__ __forceinline__ double xsqrt_rn(double a) { return __dsqrt_rn(a); }
// radii: one block per bucket, a warp per row, lane `up` folds the row against the centroid of the ancestor `up` levels
// above the bucket: Euclidean::distance(centroid, point), sequential over the dimensions (src/distance.rs:26-35)
template <typename A>
__global__ void __launch_bounds__(BT) radii_kernel(const A* __restrict__ pts, const A* __restrict__ centers, A* __restrict__ radii, uint32_t d,
                                                   uint32_t dpad, const uint32_t* __restrict__ bucket_seg, uint32_t n_internal, uint32_t levels) {
    const uint32_t b = blockIdx.x;
    const uint32_t lo = bucket_seg[b], hi = bucket_seg[b + 1];
    if (hi == lo) return;
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t h = n_internal + b;
    if (lane >= levels) return;
    const uint32_t anc = ((h + 1) >> lane) - 1;
    const A* c = centers + (uint64_t)anc * dpad;
    A best = A(0);
    for (uint32_t i = lo + warp; i < hi; i += BT / 32) {
        const A* r = pts + (uint64_t)i * dpad;
        A acc = A(0);
        for (uint32_t j = 0; j < d; ++j) {
            const A diff = c[j] - r[j];
            acc = acc + diff * diff;
        }
        const A dist = xsqrt_rn(acc);
        if (dist > best) best = dist;
    }
    atomic_max_nonneg(&radii[anc], best);
}
template <typename A>
__global__ void empty_nodes_kernel(A* __restrict__ radii, const uint32_t* __restrict__ cnt, uint32_t n_nodes) {
    const uint32_t node = blockIdx.x * blockDim.x + threadIdx.x;
    if (node < n_nodes && cnt[node] == 0) radii[node] = A(-1);
}

// ---- host driver ---------------------------------------------------------------------------------------------------
struct Scratch {
    std::vector<void*> ptrs;
    ~Scratch() { for (void* p : ptrs) cudaFree(p); }
    template <typename T> cudaError_t get(T** out, size_t count) {
        void* p = nullptr;
        cudaError_t e = cudaMalloc(&p, std::max<size_t>(count, 1) * sizeof(T));
        if (e == cudaSuccess) ptrs.push_back(p);
        *out = (T*)p;
        return e;
    }
};

static uint32_t choose_levels(uint64_t n, uint32_t bucket_size) {
    uint32_t L = 0;
    while (((n + ((uint64_t(1) << L) - 1)) >> L) > bucket_size) ++L;
    return L;
}

// the level-by-level partition of idx[0, n) (ascending on entry) for levels [0, levels) of `shape`; idx ends in idx_a
template <typename A>
static int partition_levels(const A* raw, uint64_t stride, uint32_t d, const TreeShape& shape, uint32_t levels, uint32_t* idx_a, uint32_t* idx_b,
                            const uint32_t* const* seg_dev, Scratch& sc, cudaStream_t st, std::string& err, uint32_t** idx_final,
                            uint32_t rule = 0, A* plane_w = nullptr, A* plane_t = nullptr, uint32_t plane_levels = 0, uint32_t dpad = 0) {
    using U = typename KeyT<A>::U;
    constexpr int VB = KeyT<A>::VB;
    const uint64_t n = shape.n;
    if (levels == 0) { *idx_final = idx_a; return 0; }
    const uint32_t max_seg = 1u << (levels - 1);
    // the longest segment of every level (the plain shape: ceil(n / 2^l); tile-aligned shapes split less evenly)
    std::vector<uint64_t> longest(levels, 0);
    for (uint32_t l = 0; l < levels; ++l)
        for (size_t s2 = 0; s2 + 1 < shape.seg[l].size(); ++s2) longest[l] = std::max<uint64_t>(longest[l], shape.seg[l][s2 + 1] - shape.seg[l][s2]);
    auto blocks_per_seg = [&](uint32_t l) { return (uint32_t)std::max<uint64_t>(1, (longest[l] + ROWS - 1) / ROWS); };
    size_t max_blocks = 0, max_big_seg = 0;
    for (uint32_t l = 0; l < levels; ++l) {
        max_blocks = std::max<size_t>(max_blocks, (size_t)blocks_per_seg(l) << l);
        if (longest[l] > SMALL_MAX) max_big_seg = size_t(1) << l;
    }
    U *kv = nullptr, *mn = nullptr, *mx = nullptr;
    uint32_t *col = nullptr, *hist = nullptr, *csum = nullptr, *cex = nullptr;
    SelState<U>* state = nullptr;
    GB_CU(sc.get(&kv, n));
    A* wdir = nullptr;
    // two-means rule: samples per segment bounded by 160 KB of shared memory
    const uint32_t ds = d | 1u;
    const uint32_t m_max = (uint32_t)std::min<uint64_t>(BT, std::max<uint64_t>(8, (160u * 1024u / 4u - 2u * d) / ds));
    const size_t dir_smem = ((size_t)m_max * ds + 2u * d) * sizeof(float);
    if (rule == 1) {
        GB_CU(sc.get(&wdir, (size_t)max_seg * d));
        if (dir_smem > 200u * 1024u) { err = "rows too wide for the two-means split rule"; return (int)cudaErrorInvalidValue; }
        GB_CU(allow_max_dynamic_smem(two_means_dir_kernel<A>));
    } else {
        GB_CU(sc.get(&mn, (size_t)max_seg * d));
        GB_CU(sc.get(&mx, (size_t)max_seg * d));
        GB_CU(sc.get(&col, max_seg));
    }
    GB_CU(sc.get(&state, max_seg));
    GB_CU(sc.get(&hist, std::max<size_t>(1, max_big_seg) * 256));
    GB_CU(sc.get(&csum, max_blocks));
    GB_CU(sc.get(&cex, max_blocks));
    GB_CU(cudaMemsetAsync(hist, 0, std::max<size_t>(1, max_big_seg) * 256 * 4, st));
    uint32_t *cur = idx_a, *nxt = idx_b;
    for (uint32_t l = 0; l < levels; ++l) {
        const uint32_t n_seg = 1u << l, cps = blocks_per_seg(l), nb = n_seg * cps;
        const uint32_t* seg_l = seg_dev[l];
        const uint32_t* seg_h = seg_dev[l] + 1;   // contiguous boundaries: the end of segment s is the start of s + 1
        const uint32_t* seg_n = seg_dev[l + 1];
        if (rule == 1) {
            two_means_dir_kernel<A><<<n_seg, BT, dir_smem, st>>>(raw, stride, d, cur, seg_l, seg_h, m_max, wdir);
            proj_keys_kernel<A><<<nb, BT, 0, st>>>(raw, stride, d, cur, seg_l, seg_h, cps, wdir, kv);
        } else {
            GB_CU(cudaMemsetAsync(mn, 0xff, (size_t)n_seg * d * sizeof(U), st));
            GB_CU(cudaMemsetAsync(mx, 0x00, (size_t)n_seg * d * sizeof(U), st));
            minmax_kernel<A><<<nb, BT, 0, st>>>(raw, stride, d, cur, seg_l, seg_h, cps, mn, mx);
            choose_kernel<A><<<(n_seg + 127) / 128, 128, 0, st>>>(mn, mx, d, n_seg, seg_l, seg_h, col);
            keys_kernel<A><<<nb, BT, 0, st>>>(raw, stride, cur, seg_l, seg_h, cps, col, kv);
        }
        if (longest[l] > SMALL_MAX) {
            init_state_kernel<U><<<(n_seg + 127) / 128, 128, 0, st>>>(seg_l, seg_h, n_seg, 0, state, rule == 1 ? seg_n : nullptr);
            for (int pass = 0; pass < VB + 4; ++pass) {
                hist_kernel<A><<<nb, BT, 0, st>>>(kv, cur, seg_l, seg_h, cps, state, pass, hist);
                pick_kernel<U, VB><<<(n_seg + 127) / 128, 128, 0, st>>>(hist, state, seg_l, seg_h, n_seg, pass);
            }
        } else {
            select_small_kernel<A><<<n_seg, BT, 0, st>>>(kv, cur, seg_l, seg_h, 0, state, rule == 1 ? seg_n : nullptr);
        }
        if (rule == 1 && plane_w && l < plane_levels)
            save_planes_kernel<A><<<(n_seg * dpad + 255) / 256, 256, 0, st>>>(wdir, state, seg_l, seg_h, n_seg, n_seg - 1, d, dpad, plane_w, plane_t);
        count_left_kernel<A><<<nb, BT, 0, st>>>(kv, cur, seg_l, seg_h, cps, state, csum);
        scan_blocks_kernel<<<1, 1024, 0, st>>>(csum, cex, nb);
        scatter_kernel<A><<<nb, BT, 0, st>>>(kv, cur, seg_l, seg_h, seg_n, cps, state, cex, nxt);
        GB_CU(cudaGetLastError());
        std::swap(cur, nxt);
    }
    *idx_final = cur;
    return 0;
}

static int upload_shape(const TreeShape& shape, Scratch& sc, std::vector<uint32_t*>& seg_dev, cudaStream_t st, std::string& err) {
    seg_dev.assign(shape.L + 1, nullptr);
    for (uint32_t l = 0; l <= shape.L; ++l) {
        GB_CU(sc.get(&seg_dev[l], shape.seg[l].size()));
        GB_CU(cudaMemcpyAsync(seg_dev[l], shape.seg[l].data(), shape.seg[l].size() * 4, cudaMemcpyHostToDevice, st));
    }
    return 0;
}

template <typename A>
int build_ball_tree(const A* raw, uint64_t n_all, uint32_t d, uint64_t stride, uint32_t bucket_size, uint32_t shard_depth, uint32_t shard_index,
                    TreeShape& shape, uint64_t* n_out, BallOut<A> (*alloc_out)(void* ctx, uint64_t n, const TreeShape& shape), void* ctx,
                    cudaStream_t st, std::string& err, uint32_t rule, uint32_t order_levels) {
    Scratch sc;
    uint32_t *idx_a = nullptr, *idx_b = nullptr;
    GB_CU(sc.get(&idx_a, n_all));
    GB_CU(sc.get(&idx_b, n_all));
    iota_kernel<<<(unsigned)((n_all + 255) / 256), 256, 0, st>>>(idx_a, n_all);
    GB_CU(cudaGetLastError());
    uint32_t* idx = idx_a;
    uint64_t lo = 0, n = n_all;
    if (shard_depth) {
        // the first shard_depth levels over all points; subtree shard_index is then a contiguous range of idx
        TreeShape top;
        top.init(n_all, shard_depth);
        std::vector<uint32_t*> seg_dev;
        int rc = upload_shape(top, sc, seg_dev, st, err);
        if (rc) return rc;
        rc = partition_levels<A>(raw, stride, d, top, shard_depth, idx_a, idx_b, seg_dev.data(), sc, st, err, &idx);
        if (rc) return rc;
        lo = top.seg[shard_depth][shard_index];
        n = top.seg[shard_depth][shard_index + 1] - lo;
        GB_CU(cudaStreamSynchronize(st));
    }
    *n_out = n;
    if (n == 0) return 0;
    // the shard (or everything) as a fresh problem: its rows sit at idx[lo, lo + n), ascending
    uint32_t* other = idx == idx_a ? idx_b : idx_a;
    if (lo) GB_CU(cudaMemcpyAsync(other, idx + lo, n * 4, cudaMemcpyDeviceToDevice, st));
    uint32_t* work_a = lo ? other : idx;
    uint32_t* work_b = lo ? idx : other;  // stream order: the copy above has read idx before the partition overwrites it
    if (rule == 1 && bucket_size >= TILE_ROWS && n >= 4 * TILE_ROWS) {
        // tile-aligned shape: every node of the tree starts on a multiple of 128 rows, so that a 128-row tile of the tensor
        // path's point image never straddles two buckets (a straddling tile mixes two clusters and no ball bounds it)
        uint32_t L = 0;
        for (;; ++L) {
            shape.init(n, L, TILE_ROWS);
            uint32_t longest = 0;
            for (size_t s2 = 0; s2 + 1 < shape.seg[L].size(); ++s2) longest = std::max(longest, shape.seg[L][s2 + 1] - shape.seg[L][s2]);
            if (longest <= std::max(bucket_size, 2 * TILE_ROWS) / TILE_ROWS * TILE_ROWS) break;
        }
    } else
    shape.init(n, choose_levels(n, bucket_size));
    // two-means rule: the stored order may follow `order_levels` more levels of the split than the tree has nodes for
    // (rows of a bucket grouped by the sub-clusters the next cuts would separate); the boundaries of the levels the tree
    // does have are the same in both shapes
    TreeShape order_shape;
    const bool deeper = rule == 1 && order_levels > 0 && n >= 1024;
    if (deeper) order_shape.init(n, shape.L + order_levels, shape.align);
    const TreeShape& pshape = deeper ? order_shape : shape;
    std::vector<uint32_t*> seg_dev;
    int rc = upload_shape(pshape, sc, seg_dev, st, err);
    if (rc) return rc;
    const uint32_t L = shape.L, n_internal = (1u << L) - 1, n_buckets = 1u << L, n_nodes = (1u << (L + 1)) - 1;
    const uint32_t vecn = 16 / sizeof(A), dpad = (d + vecn - 1) / vecn * vecn;
    A *plane_w = nullptr, *plane_t = nullptr;   // two-means rule: the cuts of the tree's internal nodes
    if (rule == 1 && n_internal) {
        GB_CU(sc.get(&plane_w, (size_t)n_internal * dpad));
        GB_CU(sc.get(&plane_t, (size_t)n_internal));
    }
    uint32_t* fin = nullptr;
    rc = partition_levels<A>(raw, stride, d, pshape, pshape.L, work_a, work_b, seg_dev.data(), sc, st, err, &fin, rule, plane_w, plane_t, L, dpad);
    if (rc) return rc;

    BallOut<A> out = alloc_out(ctx, n, shape);
    if (!out.pts || !out.ids || !out.centers || !out.radii) { err = "allocation of the tree arrays failed"; return (int)cudaErrorMemoryAllocation; }
    if (plane_w && out.plane_w && out.plane_t) {
        GB_CU(cudaMemcpyAsync(out.plane_w, plane_w, (size_t)n_internal * dpad * sizeof(A), cudaMemcpyDeviceToDevice, st));
        GB_CU(cudaMemcpyAsync(out.plane_t, plane_t, (size_t)n_internal * sizeof(A), cudaMemcpyDeviceToDevice, st));
    }
    gather_rows_kernel<A><<<(unsigned)((n * dpad + 255) / 256), 256, 0, st>>>(raw, stride, d, dpad, fin, n, out.pts, out.ids);
    GB_CU(cudaGetLastError());
    // per-node point counts from the shape
    std::vector<uint32_t> cnt(n_nodes);
    for (uint32_t l = 0; l <= L; ++l)
        for (uint32_t s = 0; s < (1u << l); ++s) cnt[(1u << l) - 1 + s] = shape.seg[l][s + 1] - shape.seg[l][s];
    uint32_t* cnt_dev = nullptr;
    GB_CU(sc.get(&cnt_dev, n_nodes));
    GB_CU(cudaMemcpyAsync(cnt_dev, cnt.data(), (size_t)n_nodes * 4, cudaMemcpyHostToDevice, st));
    GB_CU(cudaMemsetAsync(out.centers, 0, (size_t)n_nodes * dpad * sizeof(A), st));
    bucket_sum_kernel<A><<<n_buckets, 128, 0, st>>>(out.pts, d, dpad, seg_dev[L], n_internal, out.centers);
    for (uint32_t l = L; l-- > 0;) {
        const uint32_t first = (1u << l) - 1, count = 1u << l;
        node_sum_kernel<A><<<(unsigned)(((uint64_t)count * d + 255) / 256), 256, 0, st>>>(out.centers, first, count, d, dpad);
    }
    centroid_kernel<A><<<(unsigned)(((uint64_t)n_nodes * dpad + 255) / 256), 256, 0, st>>>(out.centers, out.radii, cnt_dev, n_nodes, d, dpad);
    radii_kernel<A><<<n_buckets, BT, 0, st>>>(out.pts, out.centers, out.radii, d, dpad, seg_dev[L], n_internal, L + 1);
    empty_nodes_kernel<A><<<(n_nodes + 255) / 256, 256, 0, st>>>(out.radii, cnt_dev, n_nodes);
    GB_CU(cudaGetLastError());
    GB_CU(cudaStreamSynchronize(st));  // cnt (host) and the scratch arrays are released on return
    return 0;
}

template int build_ball_tree<float>(const float*, uint64_t, uint32_t, uint64_t, uint32_t, uint32_t, uint32_t, TreeShape&, uint64_t*,
                                    BallOut<float> (*)(void*, uint64_t, const TreeShape&), void*, cudaStream_t, std::string&, uint32_t, uint32_t);
template int build_ball_tree<double>(const double*, uint64_t, uint32_t, uint64_t, uint32_t, uint32_t, uint32_t, TreeShape&, uint64_t*,
                                     BallOut<double> (*)(void*, uint64_t, const TreeShape&), void*, cudaStream_t, std::string&, uint32_t, uint32_t);

// ======================================================================================================================
// Vantage-point tree (create_node, src/vantage_point_tree.rs:146-197) level by level on the device.  The host builder sorts
// each slice by (distance to the vantage point, id), takes the LAST element of the sorted slice as the next vantage point,
// the first half as `near`, the rest as `far`, mu = far[0].distance.  None of that needs the sort itself:
//   vantage point of a slice = its maximum on the (distance to the parent's vantage point, id) key  -> select, rank len-1
//   near / far                = split at rank (len-1)/2 of the (distance to the vantage point, id) key -> select + partition
// Only the stored order of a bucket is the sorted order, so the buckets are sorted once at the end.  The partition places
// [near | far | vantage point] exactly as the reference's slices lie, and the keys travel with the indices so that the next
// level can pick its vantage points.
template <typename A>
__global__ void __launch_bounds__(BT) vp_keys_kernel(const A* __restrict__ raw, uint64_t stride, uint32_t d, const uint32_t* __restrict__ idx,
                                                     const uint32_t* __restrict__ seg_l, const uint32_t* __restrict__ seg_h, uint32_t cps,
                                                     const SelState<typename KeyT<A>::U>* __restrict__ st, typename KeyT<A>::U* __restrict__ kv,
                                                     uint32_t* __restrict__ vp_pos) {
    using U = typename KeyT<A>::U;
    const Span sp = block_span(seg_l, seg_h, cps);
    if (sp.cnt == 0) return;
    const uint32_t vp = st[sp.seg].pi;  // the id selected as this slice's vantage point
    const A* vrow = raw + (uint64_t)vp * stride;
    for (uint32_t r = threadIdx.x; r < sp.cnt; r += BT) {
        const uint32_t id = idx[sp.lo + r];
        if (id == vp) { kv[sp.lo + r] = ~(U)0; vp_pos[sp.seg] = sp.lo + r; continue; }   // sorts after every real distance
        const A* row = raw + (uint64_t)id * stride;
        A acc = A(0);
        for (uint32_t j = 0; j < d; ++j) {
            const A diff = row[j] - vrow[j];
            acc = acc + diff * diff;
        }
        kv[sp.lo + r] = ord_key(xsqrt_rn(acc));
    }
}
template <typename A>
__global__ void __launch_bounds__(BT) vp_scatter_kernel(const typename KeyT<A>::U* __restrict__ kv, const uint32_t* __restrict__ idx,
                                                        const uint32_t* __restrict__ seg_l, const uint32_t* __restrict__ seg_h, uint32_t cps,
                                                        const SelState<typename KeyT<A>::U>* __restrict__ st, const uint32_t* __restrict__ cex,
                                                        const uint32_t* __restrict__ vp_pos, uint32_t* __restrict__ idx_out,
                                                        typename KeyT<A>::U* __restrict__ kv_out) {
    using U = typename KeyT<A>::U;
    __shared__ uint32_t wsum[BT / 32];
    const Span sp = block_span(seg_l, seg_h, cps);
    if (sp.cnt == 0) return;
    const SelState<U> s = st[sp.seg];
    const uint32_t len = sp.seg_hi - sp.seg_lo;
    const uint32_t mid = sp.seg_lo + (len - 1) / 2;   // first position of `far`
    const uint32_t vpp = vp_pos[sp.seg];
    const uint32_t left_before = cex[blockIdx.x] - cex[sp.seg * cps];
    constexpr int PER = ROWS / BT;
    uint32_t ids[PER]; U ks[PER]; bool lf[PER];
    uint32_t mine = 0;
#pragma unroll
    for (int i = 0; i < PER; ++i) {
        const uint32_t r = threadIdx.x * PER + i;
        lf[i] = false; ids[i] = 0; ks[i] = 0;
        if (r < sp.cnt) { ids[i] = idx[sp.lo + r]; ks[i] = kv[sp.lo + r]; lf[i] = goes_left<U>(ks[i], ids[i], s); mine += lf[i] ? 1u : 0u; }
    }
    uint32_t incl = mine;
    for (int o = 1; o < 32; o <<= 1) { const uint32_t v = __shfl_up_sync(0xffffffffu, incl, o); if ((int)(threadIdx.x & 31) >= o) incl += v; }
    if ((threadIdx.x & 31) == 31) wsum[threadIdx.x >> 5] = incl;
    __syncthreads();
    uint32_t wbase = 0;
    for (uint32_t w = 0; w < (threadIdx.x >> 5); ++w) wbase += wsum[w];
    uint32_t lrun = left_before + wbase + incl - mine;
#pragma unroll
    for (int i = 0; i < PER; ++i) {
        const uint32_t r = threadIdx.x * PER + i;
        if (r >= sp.cnt) break;
        const uint32_t pos = sp.lo + r;
        uint32_t dst;
        if (pos == vpp) dst = sp.seg_hi - 1;                                              // the vantage point closes the slice
        else if (lf[i]) dst = sp.seg_lo + lrun;                                           // near, order kept
        else dst = mid + (pos - sp.seg_lo - lrun) - (pos > vpp ? 1u : 0u);               // far, order kept, the vantage point taken out
        idx_out[dst] = ids[i];
        kv_out[dst] = ks[i];
        lrun += lf[i] ? 1u : 0u;
    }
}
// node arrays: vantage point row, mu = distance key of the pivot (far[0].distance), id
template <typename A>
__global__ void vp_nodes_kernel(const A* __restrict__ raw, uint64_t stride, uint32_t d, uint32_t dpad, const SelState<typename KeyT<A>::U>* __restrict__ vsel,
                                const SelState<typename KeyT<A>::U>* __restrict__ msel, uint32_t first, uint32_t count, A* __restrict__ centers,
                                A* __restrict__ radii, uint32_t* __restrict__ vp_ids) {
    const uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= (uint64_t)count * dpad) return;
    const uint32_t s = (uint32_t)(e / dpad), j = (uint32_t)(e % dpad);
    const uint32_t vp = vsel[s].pi;
    centers[(uint64_t)(first + s) * dpad + j] = j < d ? raw[(uint64_t)vp * stride + j] : A(0);
    if (j == 0) { radii[first + s] = ord_val(msel[s].pv); vp_ids[first + s] = vp; }
}
// The index arrays ping-pong between two buffers level by level, and the slot of a vantage point belongs to no slice of
// the levels below it: the slots are written into the final buffer once more from the node array.
__global__ void vp_slots_kernel(const uint32_t* __restrict__ seg_h, uint32_t n_seg, uint32_t first, const uint32_t* __restrict__ vp_ids,
                                uint32_t* __restrict__ idx) {
    const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s < n_seg) idx[seg_h[s] - 1] = vp_ids[first + s];
}
// buckets in the reference's stored order: ascending (distance to the parent's vantage point, id); one block per bucket,
// bitonic network on the (key, id) pairs in global memory (virtual +inf pairs beyond the end never move)
template <typename A>
__global__ void __launch_bounds__(BT) vp_bucket_sort_kernel(typename KeyT<A>::U* __restrict__ kv, uint32_t* __restrict__ idx,
                                                            const uint32_t* __restrict__ seg_l, const uint32_t* __restrict__ seg_h) {
    using U = typename KeyT<A>::U;
    const uint32_t lo = seg_l[blockIdx.x], n = seg_h[blockIdx.x] - lo;
    if (n < 2) return;
    U* k = kv + lo;
    uint32_t* v = idx + lo;
    uint32_t np2 = 1;
    while (np2 < n) np2 <<= 1;
    auto cmpx = [&](uint32_t i, uint32_t j) {
        if (j > i && j < n) {
            const U ki = k[i], kj = k[j];
            const uint32_t vi = v[i], vj = v[j];
            if (ki > kj || (ki == kj && vi > vj)) { k[i] = kj; k[j] = ki; v[i] = vj; v[j] = vi; }
        }
    };
    for (uint32_t size = 2; size <= np2; size <<= 1) {
        for (uint32_t i = threadIdx.x; i < np2; i += BT) cmpx(i, i ^ (size - 1));
        __syncthreads();
        for (uint32_t stride = size >> 2; stride > 0; stride >>= 1) {
            for (uint32_t i = threadIdx.x; i < np2; i += BT) cmpx(i, i ^ stride);
            __syncthreads();
        }
    }
}

void VpShape::init(uint64_t n_, uint32_t L_) {
    n = n_; L = L_;
    lo.assign(L + 1, {}); hi.assign(L + 1, {});
    lo[0] = {0u}; hi[0] = {(uint32_t)n};
    for (uint32_t l = 0; l < L; ++l) {
        const size_t ns = size_t(1) << l;
        lo[l + 1].resize(2 * ns); hi[l + 1].resize(2 * ns);
        for (size_t s = 0; s < ns; ++s) {
            const uint32_t a = lo[l][s], b = hi[l][s], len = b - a;
            const uint32_t half = len ? (len - 1) / 2 : 0;
            lo[l + 1][2 * s] = a;            hi[l + 1][2 * s] = a + half;            // near
            lo[l + 1][2 * s + 1] = a + half; hi[l + 1][2 * s + 1] = len ? b - 1 : a; // far; the vantage point sits at b - 1
        }
    }
}

template <typename A>
int build_vp_tree(const A* raw, uint64_t n, uint32_t d, uint64_t stride, uint32_t bucket_size, VpShape& shape,
                  VpOut<A> (*alloc_out)(void* ctx, uint64_t n, const VpShape& shape), void* ctx, cudaStream_t st, std::string& err) {
    using U = typename KeyT<A>::U;
    constexpr int VB = KeyT<A>::VB;
    Scratch sc;
    shape.init(n, choose_levels(n, bucket_size));
    const uint32_t L = shape.L, n_internal = (1u << L) - 1;
    const uint32_t vecn = 16 / sizeof(A), dpad = (d + vecn - 1) / vecn * vecn;
    VpOut<A> out = alloc_out(ctx, n, shape);
    if (!out.pts || !out.ids || !out.centers || !out.radii || !out.vp_ids) { err = "allocation of the tree arrays failed"; return (int)cudaErrorMemoryAllocation; }
    uint32_t *idx_a = nullptr, *idx_b = nullptr, *vpp = nullptr, *hist = nullptr, *csum = nullptr, *cex = nullptr;
    U *kv_a = nullptr, *kv_b = nullptr;
    SelState<U>*vsel = nullptr, *msel = nullptr;
    const uint32_t max_seg = 1u << L;
    auto blocks_per_seg = [&](uint32_t l) {
        const uint64_t maxlen = (n + ((uint64_t(1) << l) - 1)) >> l;
        return (uint32_t)std::max<uint64_t>(1, (maxlen + ROWS - 1) / ROWS);
    };
    size_t max_blocks = 1, max_big_seg = 1;
    for (uint32_t l = 0; l <= L; ++l) {
        max_blocks = std::max<size_t>(max_blocks, (size_t)blocks_per_seg(l) << l);
        if (((n + ((uint64_t(1) << l) - 1)) >> l) > SMALL_MAX) max_big_seg = size_t(1) << l;
    }
    GB_CU(sc.get(&idx_a, n)); GB_CU(sc.get(&idx_b, n)); GB_CU(sc.get(&kv_a, n)); GB_CU(sc.get(&kv_b, n));
    GB_CU(sc.get(&vpp, max_seg)); GB_CU(sc.get(&vsel, max_seg)); GB_CU(sc.get(&msel, max_seg));
    GB_CU(sc.get(&hist, max_big_seg * 256)); GB_CU(sc.get(&csum, max_blocks)); GB_CU(sc.get(&cex, max_blocks));
    GB_CU(cudaMemsetAsync(hist, 0, max_big_seg * 256 * 4, st));
    GB_CU(cudaMemsetAsync(kv_a, 0, n * sizeof(U), st));   // create_root: every distance equal, so the last id is the first vantage point
    iota_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(idx_a, n);
    std::vector<uint32_t*> lo_dev(L + 1), hi_dev(L + 1);
    for (uint32_t l = 0; l <= L; ++l) {
        GB_CU(sc.get(&lo_dev[l], shape.lo[l].size())); GB_CU(sc.get(&hi_dev[l], shape.hi[l].size()));
        GB_CU(cudaMemcpyAsync(lo_dev[l], shape.lo[l].data(), shape.lo[l].size() * 4, cudaMemcpyHostToDevice, st));
        GB_CU(cudaMemcpyAsync(hi_dev[l], shape.hi[l].data(), shape.hi[l].size() * 4, cudaMemcpyHostToDevice, st));
    }
    auto select = [&](const U* kv, const uint32_t* idx, uint32_t l, int mode, SelState<U>* state) {
        const uint32_t n_seg = 1u << l, cps = blocks_per_seg(l), nb = n_seg * cps;
        if (((n + ((uint64_t(1) << l) - 1)) >> l) > SMALL_MAX) {
            init_state_kernel<U><<<(n_seg + 127) / 128, 128, 0, st>>>(lo_dev[l], hi_dev[l], n_seg, mode, state);
            for (int pass = 0; pass < VB + 4; ++pass) {
                hist_kernel<A><<<nb, BT, 0, st>>>(kv, idx, lo_dev[l], hi_dev[l], cps, state, pass, hist);
                pick_kernel<U, VB><<<(n_seg + 127) / 128, 128, 0, st>>>(hist, state, lo_dev[l], hi_dev[l], n_seg, pass);
            }
        } else {
            select_small_kernel<A><<<n_seg, BT, 0, st>>>(kv, idx, lo_dev[l], hi_dev[l], mode, state);
        }
    };
    uint32_t *cur = idx_a, *nxt = idx_b;
    U *kcur = kv_a, *knxt = kv_b;
    for (uint32_t l = 0; l < L; ++l) {
        const uint32_t n_seg = 1u << l, cps = blocks_per_seg(l), nb = n_seg * cps, first = n_seg - 1;
        select(kcur, cur, l, 1, vsel);                                                    // the slice's last element in sorted order
        vp_keys_kernel<A><<<nb, BT, 0, st>>>(raw, stride, d, cur, lo_dev[l], hi_dev[l], cps, vsel, kcur, vpp);
        select(kcur, cur, l, 2, msel);                                                    // far[0]
        vp_nodes_kernel<A><<<(unsigned)(((uint64_t)n_seg * dpad + 255) / 256), 256, 0, st>>>(raw, stride, d, dpad, vsel, msel, first, n_seg, out.centers,
                                                                                             out.radii, out.vp_ids);
        count_left_kernel<A><<<nb, BT, 0, st>>>(kcur, cur, lo_dev[l], hi_dev[l], cps, msel, csum);
        scan_blocks_kernel<<<1, 1024, 0, st>>>(csum, cex, nb);
        vp_scatter_kernel<A><<<nb, BT, 0, st>>>(kcur, cur, lo_dev[l], hi_dev[l], cps, msel, cex, vpp, nxt, knxt);
        GB_CU(cudaGetLastError());
        std::swap(cur, nxt); std::swap(kcur, knxt);
    }
    for (uint32_t l = 0; l < L; ++l)
        vp_slots_kernel<<<((1u << l) + 127) / 128, 128, 0, st>>>(hi_dev[l], 1u << l, (1u << l) - 1, out.vp_ids, cur);
    vp_bucket_sort_kernel<A><<<1u << L, BT, 0, st>>>(kcur, cur, lo_dev[L], hi_dev[L]);
    gather_rows_kernel<A><<<(unsigned)((n * dpad + 255) / 256), 256, 0, st>>>(raw, stride, d, dpad, cur, n, out.pts, out.ids);
    GB_CU(cudaGetLastError());
    GB_CU(cudaStreamSynchronize(st));
    (void)n_internal;
    return 0;
}
template int build_vp_tree<float>(const float*, uint64_t, uint32_t, uint64_t, uint32_t, VpShape&, VpOut<float> (*)(void*, uint64_t, const VpShape&), void*,
                                  cudaStream_t, std::string&);
template int build_vp_tree<double>(const double*, uint64_t, uint32_t, uint64_t, uint32_t, VpShape&, VpOut<double> (*)(void*, uint64_t, const VpShape&),
                                   void*, cudaStream_t, std::string&);

// ---- centre and range of the stored points for the tensor path --------------------------------------------------------
constexpr uint32_t CH_ROWS = 4096;
__global__ void chunk_sums_kernel(const float* __restrict__ pts, uint64_t n, uint32_t d, uint32_t dpad, double* __restrict__ part) {
    const uint32_t ch = blockIdx.x;
    const uint64_t lo = (uint64_t)ch * CH_ROWS, hi = min(n, lo + CH_ROWS);
    for (uint32_t j = threadIdx.x; j < d; j += blockDim.x) {
        double m = 0.0;
        for (uint64_t i = lo; i < hi; ++i) m += (double)pts[i * dpad + j];
        part[(uint64_t)ch * dpad + j] = m;
    }
}
__global__ void mean_kernel(const double* __restrict__ part, uint32_t n_ch, uint64_t n, uint32_t d, uint32_t dpad, float* __restrict__ center) {
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= dpad) return;
    double m = 0.0;
    if (j < d) for (uint32_t c = 0; c < n_ch; ++c) m += part[(uint64_t)c * dpad + j];
    center[j] = j < d ? (float)(m / (double)n) : 0.f;
}
__global__ void maxabs_kernel(const float* __restrict__ pts, uint64_t n, uint32_t d, uint32_t dpad, const float* __restrict__ center,
                              unsigned int* __restrict__ out_bits) {
    float m = 0.f;
    const uint64_t total = n * dpad;
    for (uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t j = (uint32_t)(e % dpad);
        if (j < d) m = fmaxf(m, fabsf(pts[e] - center[j]));
    }
    for (int o = 16; o; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0) atomicMax(out_bits, __float_as_uint(m));
}
int centre_and_range_f32(const float* pts, uint64_t n, uint32_t d, uint32_t dpad, float* center_dev, float* center_host, float* maxabs,
                         cudaStream_t st, std::string& err) {
    Scratch sc;
    const uint32_t n_ch = (uint32_t)((n + CH_ROWS - 1) / CH_ROWS);
    double* part = nullptr;
    unsigned int* bits = nullptr;
    GB_CU(sc.get(&part, (size_t)n_ch * dpad));
    GB_CU(sc.get(&bits, 1));
    GB_CU(cudaMemsetAsync(bits, 0, 4, st));
    chunk_sums_kernel<<<n_ch, 128, 0, st>>>(pts, n, d, dpad, part);
    mean_kernel<<<(dpad + 127) / 128, 128, 0, st>>>(part, n_ch, n, d, dpad, center_dev);
    maxabs_kernel<<<1184, 256, 0, st>>>(pts, n, d, dpad, center_dev, bits);
    GB_CU(cudaGetLastError());
    unsigned int hb = 0;
    GB_CU(cudaMemcpyAsync(&hb, bits, 4, cudaMemcpyDeviceToHost, st));
    GB_CU(cudaMemcpyAsync(center_host, center_dev, (size_t)dpad * 4, cudaMemcpyDeviceToHost, st));
    GB_CU(cudaStreamSynchronize(st));
    memcpy(maxabs, &hb, 4);
    return 0;
}

}  // namespace gb
}  // namespace petal
