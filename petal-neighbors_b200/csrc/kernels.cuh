// kernels.cuh -- sm_100a device code of the exact k-NN / radius engine.
//
// Replaces, for batches of queries, the per-query recursion of the reference:
//   knn_tile_kernel   : nearest_k_neighbors_in_subtree src/ball_tree.rs:203-243,
//                       nearest_neighbor_in_subtree :149-196, search_node
//                       src/vantage_point_tree.rs:100-130 (k = 1)
//   radius_kernel     : neighbors_within_radius_in_subtree src/ball_tree.rs:250-294
//   merge_lists_kernel: BinaryHeap::into_sorted_vec :117 for split scans / point shards
// Every distance is Euclidean::distance (src/distance.rs:26-35) evaluated with explicit
// round-to-nearest intrinsics in the reference's order (sub, mul, add per dimension, then
// sqrt) so that it is bit-identical to the Rust fold: the compiler can neither contract the
// multiply-add into an FMA nor reassociate the sum.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <float.h>

namespace petal {

constexpr int TQ = 128;           // queries per CTA of the tile scan, one per thread
constexpr int RP = 8;             // points per register tile (independent fold chains per thread)
constexpr int TILE_BYTES = 16384; // one shared-memory point tile (two are in flight)
constexpr int MAX_STACK = 40;     // traversal stack depth (tree depth <= 32)
constexpr uint32_t NO_ID = 0xFFFFFFFFu;

template <typename A> struct VT;
template <> struct VT<float>  { using V = float4;  static constexpr int N = 4; };
template <> struct VT<double> { using V = double2; static constexpr int N = 2; };

// ---- exact IEEE arithmetic (never contracted, never reassociated) -------------------------
__device__ __forceinline__ float  xsub(float a, float b)   { return __fsub_rn(a, b); }
__device__ __forceinline__ float  xmul(float a, float b)   { return __fmul_rn(a, b); }
__device__ __forceinline__ float  xadd(float a, float b)   { return __fadd_rn(a, b); }
__device__ __forceinline__ float  xsqrt(float a)           { return __fsqrt_rn(a); }
__device__ __forceinline__ double xsub(double a, double b) { return __dsub_rn(a, b); }
__device__ __forceinline__ double xmul(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double xadd(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double xsqrt(double a)          { return __dsqrt_rn(a); }

template <typename A> __device__ __forceinline__ A pos_inf();
template <> __device__ __forceinline__ float  pos_inf<float>()  { return __int_as_float(0x7f800000); }
template <> __device__ __forceinline__ double pos_inf<double>() { return __longlong_as_double(0x7ff0000000000000LL); }

// one vector step of the sequential fold: sum += (q_j - p_j)^2 for the 4 (2) dims of a V
__device__ __forceinline__ float fold(float acc, const float4& q, const float4& p) {
    float t;
    t = xsub(q.x, p.x); acc = xadd(acc, xmul(t, t));
    t = xsub(q.y, p.y); acc = xadd(acc, xmul(t, t));
    t = xsub(q.z, p.z); acc = xadd(acc, xmul(t, t));
    t = xsub(q.w, p.w); acc = xadd(acc, xmul(t, t));
    return acc;
}
__device__ __forceinline__ double fold(double acc, const double2& q, const double2& p) {
    double t;
    t = xsub(q.x, p.x); acc = xadd(acc, xmul(t, t));
    t = xsub(q.y, p.y); acc = xadd(acc, xmul(t, t));
    return acc;
}

__device__ __forceinline__ float4  vzero(float)  { return make_float4(0.f, 0.f, 0.f, 0.f); }
__device__ __forceinline__ double2 vzero(double) { return make_double2(0., 0.); }

// Conservative squared-domain acceptance threshold: any s with sqrt_rn(s) <= kth satisfies
// s <= thresh2(kth).  (All comparisons of the reference are on sqrt'd distances, SURVEY S4; the
// cheap squared test only filters, the exact test runs on the sqrt'd value.)
__device__ __forceinline__ float  thresh2(float kth)  { return xadd(xmul(xmul(kth, kth), 1.00000095367431640625f), FLT_MIN); }
__device__ __forceinline__ double thresh2(double kth) { return xadd(xmul(xmul(kth, kth), 1.0 + 1.7763568394002505e-15), DBL_MIN); }

// ---- TMA 1-D bulk copy global -> shared, completion on an mbarrier (leaf buckets are contiguous,
// 16-byte aligned spans, so no tensor map is needed) ------------------------------------------
__device__ __forceinline__ uint32_t smem_addr_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void bulk_bar_init(uint64_t* bar) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_addr_u32(bar)));
}
__device__ __forceinline__ void bulk_load(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_addr_u32(bar)), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_addr_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_addr_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void bulk_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred P1;\n\t"
        "BW_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1, %2;\n\t"
        "@P1 bra BW_DONE;\n\t"
        "bra BW_LOOP;\n\t"
        "BW_DONE:\n\t"
        "}" ::"r"(smem_addr_u32(bar)), "r"(parity), "r"(100000u) : "memory");
}

// ---- flattened tree as seen by the device --------------------------------------------------
template <typename A>
struct DevTree {
    const typename VT<A>::V* pts;  // n x dpad, bucket order
    const uint32_t* ids;           // n
    const uint32_t* bucket_lo;
    const uint32_t* bucket_hi;
    const typename VT<A>::V* centers;  // n_nodes x dpad
    const A* radii;                // ball: radius (-1 empty) ; vp: mu
    const uint32_t* vp_ids;        // vp only
    uint32_t n, d, dpad, dv;       // dv = dpad / VT<A>::N
    uint32_t L, n_internal, n_buckets, n_nodes;
    int kind;
    A slack;                       // (2d + 8) * unit roundoff: relative slack of a triangle bound
    // two-means partition only (else null): the cut of every internal node -- direction (n_internal x dpad) and pivot key;
    // a row with  row . w < t  went to the left child.  Used to route queries to their home bucket, nothing else.
    const A* plane_w;
    const A* plane_t;
};

// ---- per-thread running top-k in registers (Neighbor + BinaryHeap, src/ball_tree.rs:378-423,
// :109, :219-225), kept sorted ascending by (distance, index).  The list always has K slots; for
// k < K the first K-k slots hold (-inf, 0) sentinels that nothing can displace, so the current
// k-th best is ALWAYS slot K-1 and every register index is static (a runtime slot index would
// push the arrays to local memory).  Results are slots [K-k, K). ------------------------------
template <typename A, int K>
struct TopK {
    A kd[K];
    uint32_t ki[K];
    A t2;           // thresh2(kth): squared-domain acceptance filter
    A fd;           // floor key for multi-pass k > K: only keys > (fd, fi) are accepted
    uint32_t fi;
    bool has_floor;

    __device__ __forceinline__ A kth() const { return kd[K - 1]; }

    __device__ __forceinline__ void init(bool active, uint32_t k) {
#pragma unroll
        for (int i = 0; i < K; ++i) {
            const bool real = i >= K - (int)k;
            kd[i] = real ? pos_inf<A>() : -pos_inf<A>();
            ki[i] = real ? NO_ID : 0u;
        }
        t2 = active ? pos_inf<A>() : A(-1);
        has_floor = false; fd = A(0); fi = 0;
    }
    __device__ __forceinline__ void set_floor(A d, uint32_t i) { has_floor = true; fd = d; fi = i; }

    // exact test + insertion on the sqrt'd distance
    __device__ __forceinline__ void offer(A d, uint32_t id) {
        if (has_floor && !(d > fd || (d == fd && id > fi))) return;
        if (!(d < kd[K - 1] || (d == kd[K - 1] && id < ki[K - 1]))) return;
        kd[K - 1] = d; ki[K - 1] = id;
#pragma unroll
        for (int i = K - 1; i > 0; --i) {
            const bool sw = (kd[i] < kd[i - 1]) || (kd[i] == kd[i - 1] && ki[i] < ki[i - 1]);
            const A lo_d = sw ? kd[i] : kd[i - 1], hi_d = sw ? kd[i - 1] : kd[i];
            const uint32_t lo_i = sw ? ki[i] : ki[i - 1], hi_i = sw ? ki[i - 1] : ki[i];
            kd[i - 1] = lo_d; kd[i] = hi_d; ki[i - 1] = lo_i; ki[i] = hi_i;
        }
        t2 = thresh2(kd[K - 1]);
    }
    __device__ __forceinline__ void offer_sq(A s, uint32_t id) { offer(xsqrt(s), id); }

    // results: slot K-k+i -> out[i]
    __device__ __forceinline__ void store(A* out_d, uint32_t* out_i, uint32_t k) const {
#pragma unroll
        for (int i = 0; i < K; ++i)
            if (i >= K - (int)k) { out_d[i - (K - (int)k)] = kd[i]; out_i[i - (K - (int)k)] = ki[i]; }
    }
};

// ---- the same container with runtime-indexed arrays, i.e. deliberately in thread-local memory (L1):
// the tile scan touches its list only on the rare accepted candidate (~k ln(N/k) times per query)
// while its hot loop is bound by instruction issue, so registers are worth more as occupancy.
template <typename A, int K>
struct TopKLocal {
    A kd[K];
    uint32_t ki[K];
    A t2, fd, kth_d;
    uint32_t fi, kth_i, k;
    bool has_floor;
    __device__ __forceinline__ A kth() const { return kth_d; }
    __device__ __forceinline__ void init(bool active, uint32_t k_) {
        k = k_;
#pragma unroll 1
        for (uint32_t i = 0; i < k; ++i) { kd[i] = pos_inf<A>(); ki[i] = NO_ID; }
        kth_d = pos_inf<A>(); kth_i = NO_ID;
        t2 = active ? pos_inf<A>() : A(-1);
        has_floor = false; fd = A(0); fi = 0;
    }
    __device__ __forceinline__ void set_floor(A d, uint32_t i) { has_floor = true; fd = d; fi = i; }
    __device__ __noinline__ void offer(A d, uint32_t id) {
        if (has_floor && !(d > fd || (d == fd && id > fi))) return;
        if (!(d < kth_d || (d == kth_d && id < kth_i))) return;
        uint32_t p = k - 1;
#pragma unroll 1
        while (p > 0) {
            const A pd = kd[p - 1];
            const uint32_t pi = ki[p - 1];
            if (!(d < pd || (d == pd && id < pi))) break;
            kd[p] = pd; ki[p] = pi;
            --p;
        }
        kd[p] = d; ki[p] = id;
        kth_d = kd[k - 1]; kth_i = ki[k - 1];
        t2 = thresh2(kth_d);
    }
    __device__ __forceinline__ void offer_sq(A s, uint32_t id) { offer(xsqrt(s), id); }
    __device__ __forceinline__ void store(A* out_d, uint32_t* out_i, uint32_t) const {
#pragma unroll 1
        for (uint32_t i = 0; i < k; ++i) { out_d[i] = kd[i]; out_i[i] = ki[i]; }
    }
};
// small d (DVR 1-2: pruned, few thousand pairs per query, insert-heavy) -> registers; otherwise local
template <typename A, int K, int DVR> struct TileTopK { using type = TopKLocal<A, K>; };
template <typename A, int K> struct TileTopK<A, K, 1> { using type = TopK<A, K>; };
template <typename A, int K> struct TileTopK<A, K, 2> { using type = TopK<A, K>; };
template <typename A, int DVR> struct TileTopK<A, 1, DVR> { using type = TopK<A, 1>; };
template <typename A> struct TileTopK<A, 1, 1> { using type = TopK<A, 1>; };
template <typename A> struct TileTopK<A, 1, 2> { using type = TopK<A, 1>; };

// ---- block-wide counts of up to four predicates with ONE barrier ---------------------------
struct VoteBuf { uint32_t v[2][TQ / 32][4]; };
__device__ __forceinline__ void block_counts(VoteBuf& vb, int& parity, bool a, bool b, bool c, bool d,
                                             int& na, int& nb, int& nc, int& nd) {
    const unsigned full = 0xffffffffu;
    unsigned ba = __ballot_sync(full, a), bb = __ballot_sync(full, b);
    unsigned bc = __ballot_sync(full, c), bd = __ballot_sync(full, d);
    const int warp = threadIdx.x >> 5;
    if ((threadIdx.x & 31) == 0) {
        vb.v[parity][warp][0] = __popc(ba); vb.v[parity][warp][1] = __popc(bb);
        vb.v[parity][warp][2] = __popc(bc); vb.v[parity][warp][3] = __popc(bd);
    }
    __syncthreads();
    na = nb = nc = nd = 0;
#pragma unroll
    for (int w = 0; w < TQ / 32; ++w) {
        na += vb.v[parity][w][0]; nb += vb.v[parity][w][1];
        nc += vb.v[parity][w][2]; nd += vb.v[parity][w][3];
    }
    parity ^= 1;
}

template <typename A>
struct KnnArgs {
    DevTree<A> t;
    const typename VT<A>::V* q;  // nq x dpad, zero padded
    const uint32_t* qorder;      // sorted slot -> query id (tile coherence), may be null
    uint32_t nq, k;
    uint32_t split_level;        // grid.y = 2^split_level subtrees scanned independently
    A* part_d;                   // [n_splits][nq][k]
    uint32_t* part_i;
    const A* floor_d;            // optional [nq] floor keys (multi-pass k > K)
    const uint32_t* floor_i;
    unsigned long long* counters;  // [0] pairs, [1] node visits
    // split scans only (may be null): per query, the smallest k-th distance any split's list has reached so far.  It is
    // an upper bound of the final k-th distance, so every split may prune with it (strictly: lb > bound); without it a
    // split far from the query starts from +inf and walks its whole subtree's near side before its own list is full.
    A* g_bound;                  // [nq] by query id, initialised to a huge finite value
};
__device__ __forceinline__ void publish_bound(float* p, float v) { atomicMin(reinterpret_cast<int*>(p), __float_as_int(v)); }
__device__ __forceinline__ void publish_bound(double* p, double v) { atomicMin(reinterpret_cast<long long*>(p), __double_as_longlong(v)); }

// ---- the tile scan: one CTA = 128 queries (one per thread), DFS over the flattened tree with
// block-uniform control flow, buckets staged through shared memory with 16-byte loads, every
// lane folding RP independent point distances per step -------------------------------------
template <typename A, int DVR, int K, int KIND>
__global__ void __launch_bounds__(TQ) knn_tile_kernel(const KnnArgs<A> a) {
    using V = typename VT<A>::V;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    V* ps0 = reinterpret_cast<V*>(smem_raw);                    // tile buffers 0 / 1
    V* qs = reinterpret_cast<V*>(smem_raw + 2 * TILE_BYTES);    // generic-d only: [dv][TQ]
    __shared__ VoteBuf votes;
    __shared__ __align__(8) uint64_t tile_bar[2];
    __shared__ unsigned long long s_pairs, s_visits;

    const DevTree<A>& t = a.t;
    const int tid = threadIdx.x;
    const uint32_t slot = blockIdx.x * TQ + tid;
    const bool active = slot < a.nq;
    const uint32_t qid = active ? (a.qorder ? a.qorder[slot] : slot) : 0;
    const int DV = DVR > 0 ? DVR : (int)t.dv;
    const uint32_t k = a.k;
    if (tid == 0) {
        s_pairs = 0; s_visits = 0;
        bulk_bar_init(&tile_bar[0]); bulk_bar_init(&tile_bar[1]);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }

    // DVR > 0: query in registers; DVR == 0: query in a transposed smem copy; DVR < 0 ("wide" rows,
    // more than 1024 bytes): nothing is staged, query and point rows are read through L1/L2
    constexpr bool WIDE = DVR < 0;
    const V* qrow = a.q + (size_t)qid * DV;
    V qreg[DVR > 0 ? DVR : 1];
    if (DVR > 0) {
#pragma unroll
        for (int jc = 0; jc < (DVR > 0 ? DVR : 1); ++jc)
            qreg[jc] = active ? a.q[(size_t)qid * DV + jc] : vzero(A(0));
    } else if (!WIDE) {
        for (int jc = 0; jc < DV; ++jc) qs[jc * TQ + tid] = active ? a.q[(size_t)qid * DV + jc] : vzero(A(0));
    }
    __syncthreads();

    typename TileTopK<A, K, DVR>::type topk;
    topk.init(active, k);
    if (a.floor_d && active) topk.set_floor(a.floor_d[qid], a.floor_i[qid]);
    // pruning bound: this split's own k-th distance, or a smaller one another split of the same query has published
    A* const gb = a.g_bound && active ? a.g_bound + qid : nullptr;
    auto bound = [&]() -> A {
        const A own = topk.kth();
        if (!gb) return own;
        const A g = __ldcg(gb);
        return own < g ? own : g;
    };
    auto publish = [&]() {
        if (gb) { const A own = topk.kth(); if (own < __ldcg(gb)) publish_bound(gb, own); }
    };

    unsigned long long my_pairs = 0, my_visits = 0;
    int parity = 0;

    // squared fold distance from this thread's query to a row of `centers` / `pts` in global memory
    auto dist_to = [&](const V* row) -> A {
        A acc = A(0);
        if (DVR > 0) {
#pragma unroll
            for (int jc = 0; jc < (DVR > 0 ? DVR : 1); ++jc) acc = fold(acc, qreg[jc], __ldg(row + jc));
        } else if (WIDE) {
            for (int jc = 0; jc < DV; ++jc) acc = fold(acc, __ldg(qrow + jc), __ldg(row + jc));
        } else {
            for (int jc = 0; jc < DV; ++jc) acc = fold(acc, qs[jc * TQ + tid], __ldg(row + jc));
        }
        return xsqrt(acc);
    };

    // leaf loops src/ball_tree.rs:162-173, 217-226: all points of bucket b against all 128 queries
    const int TP = max(RP, (int)(TILE_BYTES / (t.dpad * sizeof(A))) / RP * RP);  // unused by the wide variant
    // Tiles are staged by TMA bulk copies (cp.async.bulk, one elected thread) into two buffers: the copy
    // of tile i+1 overlaps the distance folds on tile i; one barrier per tile protects buffer reuse.
    uint32_t tile_use[2] = {0, 0};  // uses of each buffer so far (block-uniform) -> mbarrier phase parity
    auto scan_bucket = [&](uint32_t b, bool need) {
        const uint32_t lo = t.bucket_lo[b], hi = t.bucket_hi[b];
        if (hi <= lo) return;
        const bool warp_need = __any_sync(0xffffffffu, need);
        if (WIDE) {  // all lanes read the same point row (one broadcast transaction), each its own query row
            if (warp_need) {
                if (active) my_pairs += hi - lo;
                for (uint32_t p0 = lo; p0 < hi; p0 += RP) {
                    A acc[RP];
#pragma unroll
                    for (int r = 0; r < RP; ++r) acc[r] = A(0);
                    for (int jc = 0; jc < DV; ++jc) {
                        const V qv = __ldg(qrow + jc);
#pragma unroll
                        for (int r = 0; r < RP; ++r) acc[r] = fold(acc[r], qv, __ldg(t.pts + (size_t)min(p0 + r, hi - 1) * DV + jc));
                    }
#pragma unroll
                    for (int r = 0; r < RP; ++r)
                        if (p0 + r < hi && acc[r] <= topk.t2) topk.offer_sq(acc[r], __ldg(t.ids + p0 + r));
                }
            }
            return;
        }
        const uint32_t row_bytes = t.dpad * (uint32_t)sizeof(A);
        const uint32_t n_tiles = (hi - lo + TP - 1) / TP;
        auto issue = [&](uint32_t i) {  // tid == 0 only
            const uint32_t p0 = lo + i * TP;
            const uint32_t np = min(hi - p0, (uint32_t)TP);
            bulk_load(reinterpret_cast<unsigned char*>(ps0) + (i & 1u) * TILE_BYTES, t.pts + (size_t)p0 * DV, np * row_bytes, &tile_bar[i & 1u]);
        };
        if (tid == 0) { issue(0); if (n_tiles > 1) issue(1); }
        for (uint32_t i = 0; i < n_tiles; ++i) {
            const uint32_t p0 = lo + i * TP;
            const int np = (int)min(hi - p0, (uint32_t)TP);
            const uint32_t bsel = i & 1u;
            const V* ps = reinterpret_cast<const V*>(reinterpret_cast<const unsigned char*>(ps0) + bsel * TILE_BYTES);
            bulk_wait(&tile_bar[bsel], tile_use[bsel] & 1u);
            ++tile_use[bsel];
            if (warp_need) {
                if (active) my_pairs += np;
                for (int pp = 0; pp < np; pp += RP) {
                    A acc[RP];
#pragma unroll
                    for (int r = 0; r < RP; ++r) acc[r] = A(0);
                    if (DVR > 0) {
#pragma unroll
                        for (int jc = 0; jc < (DVR > 0 ? DVR : 1); ++jc) {
#pragma unroll
                            for (int r = 0; r < RP; ++r) acc[r] = fold(acc[r], qreg[jc], ps[(pp + r) * DVR + jc]);
                        }
                    } else {
                        for (int jc = 0; jc < DV; ++jc) {
                            const V qv = qs[jc * TQ + tid];
#pragma unroll
                            for (int r = 0; r < RP; ++r) acc[r] = fold(acc[r], qv, ps[(pp + r) * DV + jc]);
                        }
                    }
#pragma unroll
                    for (int r = 0; r < RP; ++r) {
                        if (pp + r < np && acc[r] <= topk.t2)
                            topk.offer_sq(acc[r], __ldg(t.ids + p0 + pp + r));
                    }
                }
            }
            __syncthreads();  // everyone is done with this buffer: it may be refilled
            if (tid == 0 && i + 2 < n_tiles) issue(i + 2);
        }
    };

    uint32_t stack[MAX_STACK];
    int sp = 0;
    const uint32_t root = ((1u << a.split_level) - 1u) + blockIdx.y;

    if (KIND == 0) {
        // ---- ball tree: prune a node for a query iff its conservative lower bound
        // cd - R - slack*(cd+R) exceeds the query's current k-th distance (:212, strict) ----
        stack[sp++] = root;
        while (sp) {
            const uint32_t node = stack[--sp];
            ++my_visits;
            if (node >= t.n_internal) {
                const A R = t.radii[node];
                if (R < A(0)) continue;  // empty
                const A cd = dist_to(t.centers + (size_t)node * DV);
                const A lb = xsub(xsub(cd, R), xmul(t.slack, xadd(cd, R)));
                const bool need = active && !(lb > bound());
                if (!__syncthreads_or(need)) continue;
                scan_bucket(node - t.n_internal, need);
                publish();
            } else {
                const uint32_t c1 = 2 * node + 1, c2 = c1 + 1;
                const A R1 = t.radii[c1], R2 = t.radii[c2];
                A lb1 = pos_inf<A>(), lb2 = pos_inf<A>();
                if (!(R1 < A(0))) { const A cd = dist_to(t.centers + (size_t)c1 * DV); lb1 = xsub(xsub(cd, R1), xmul(t.slack, xadd(cd, R1))); }
                if (!(R2 < A(0))) { const A cd = dist_to(t.centers + (size_t)c2 * DV); lb2 = xsub(xsub(cd, R2), xmul(t.slack, xadd(cd, R2))); }
                const A bnd = bound();
                const bool need1 = active && !(R1 < A(0)) && !(lb1 > bnd);
                const bool need2 = active && !(R2 < A(0)) && !(lb2 > bnd);
                int n1, n2, npref, nany;
                block_counts(votes, parity, need1, need2, (need1 || need2) && (lb1 < lb2), need1 || need2, n1, n2, npref, nany);
                // nearer child first (:232-236), decided by the tile's majority
                const bool first1 = 2 * npref >= nany;
                const uint32_t first = first1 ? c1 : c2, second = first1 ? c2 : c1;
                const int nfirst = first1 ? n1 : n2, nsecond = first1 ? n2 : n1;
                if (nsecond) stack[sp++] = second;
                if (nfirst) stack[sp++] = first;
            }
        }
    } else {
        // ---- vantage-point tree (search_node, src/vantage_point_tree.rs:100-130): the bound of a
        // subtree is the max over its ancestors of |d(q,vp) - mu| on the far/near side ----
        A lbs[MAX_STACK];
        if (a.split_level > 0 && blockIdx.y == 0) {
            // vantage points above the split level belong to no split's subtree
            for (uint32_t node = 0; node < ((1u << a.split_level) - 1u); ++node) {
                const A dq = dist_to(t.centers + (size_t)node * DV);
                if (active) topk.offer(dq, t.vp_ids[node]);
            }
        }
        stack[sp] = root; lbs[sp] = A(0); ++sp;
        while (sp) {
            --sp;
            const uint32_t node = stack[sp];
            const A lb = lbs[sp];
            ++my_visits;
            const A bnd = bound();
            const bool need = active && !(lb > bnd);
            if (node >= t.n_internal) {
                if (!__syncthreads_or(need)) continue;
                scan_bucket(node - t.n_internal, need);
                publish();
            } else {
                const A mu = t.radii[node];
                const A dq = dist_to(t.centers + (size_t)node * DV);
                if (need) topk.offer(dq, t.vp_ids[node]);  // the vantage point is a data point (:106-109)
                const A s = xmul(t.slack, xadd(dq, mu));
                const A lbn = fmax(lb, xsub(xsub(dq, mu), s));   // near side: d(p,vp) <= mu
                const A lbf = fmax(lb, xsub(xsub(mu, dq), s));   // far side:  d(p,vp) >= mu
                const A own = topk.kth();   // the vantage point may just have tightened this split's list
                const A bnd2 = own < bnd ? own : bnd;
                const bool needn = active && !(lbn > bnd2);
                const bool needf = active && !(lbf > bnd2);
                int nn, nf, npref, nany;
                block_counts(votes, parity, needn, needf, (needn || needf) && (dq < mu), needn || needf, nn, nf, npref, nany);
                const bool near_first = 2 * npref >= nany;  // :111 `distance < radius` -> near first
                const uint32_t cn = 2 * node + 1, cf = cn + 1;
                if (near_first) {
                    if (nf) { stack[sp] = cf; lbs[sp] = lbf; ++sp; }
                    if (nn) { stack[sp] = cn; lbs[sp] = lbn; ++sp; }
                } else {
                    if (nn) { stack[sp] = cn; lbs[sp] = lbn; ++sp; }
                    if (nf) { stack[sp] = cf; lbs[sp] = lbf; ++sp; }
                }
            }
        }
    }

    if (active) {
        const size_t base = ((size_t)blockIdx.y * a.nq + qid) * k;
        topk.store(a.part_d + base, a.part_i + base, k);
    }
    if (a.counters) {
        atomicAdd(&s_pairs, my_pairs);
        if (tid == 0) s_visits = my_visits;
        __syncthreads();
        if (tid == 0) { atomicAdd(&a.counters[0], s_pairs); atomicAdd(&a.counters[1], s_visits); }
    }
}

// ---- the warp scan: ONE WARP PER QUERY, for narrow rows (dv <= 4: f32 d <= 16, f64 d <= 8) where the ball bounds prune
// almost everything and a query needs a handful of buckets.  The tile scan above walks the UNION of what its 128 queries
// need, one node after the other: fine when a batch is dense in the tree (a tile's queries share their buckets), a
// long serial chain when it is not (4096 queries on a 10M x 3 tree: 21.7 ms, against 11 ms for 262 144).  Here every
// query walks its own path (BallTree::nearest_k_neighbors_in_subtree, src/ball_tree.rs:203-243): nearer child first,
// a node is skipped iff its conservative lower bound exceeds the current k-th distance (strict, :212); the lanes fold
// the points of a bucket 32 at a time and the sorted top-k list lives across the lanes (lane i = i-th best, up to 32 per
// pass), keyed on (sqrt'd distance, index) like every other list of the engine.  Results go straight to the output
// rows: no splits, no merge.
template <typename A>
struct WarpKnnArgs {
    DevTree<A> t;
    const typename VT<A>::V* q;    // nq x dpad, zero padded
    const uint32_t* qorder;        // sorted slot -> query id (cache locality between neighbouring warps), may be null
    const uint32_t* row_map;       // query id -> output row (self query: the stored point's original index), may be null
    uint32_t nq, k;                // k <= 32 per pass
    uint64_t* out_i;
    A* out_d;
    uint32_t out_stride, out_off;
    A* floor_d;                    // [nq] (multi-pass k > 32): in = the last key of the previous pass (pass > 0), out = this pass's
    uint32_t* floor_i;
    uint32_t pass;
    unsigned long long* counters;  // [0] pairs, [1] node visits
};
template <typename A>
__global__ void __launch_bounds__(256) knn_warp_kernel(const WarpKnnArgs<A> a) {
    using V = typename VT<A>::V;
    const DevTree<A>& t = a.t;
    const int lane = threadIdx.x & 31;
    const uint32_t slot = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (slot >= a.nq) return;
    const uint32_t qid = a.qorder ? a.qorder[slot] : slot;
    const unsigned full = 0xffffffffu;
    const int DV = (int)t.dv;   // <= 4
    V qreg[4];
#pragma unroll
    for (int jc = 0; jc < 4; ++jc) qreg[jc] = jc < DV ? __ldg(a.q + (size_t)qid * DV + jc) : vzero(A(0));
    auto dist2_to = [&](const V* row) -> A {
        A acc = A(0);
#pragma unroll
        for (int jc = 0; jc < 4; ++jc)
            if (jc < DV) acc = fold(acc, qreg[jc], __ldg(row + jc));
        return acc;
    };
    // the list: lane i holds the i-th best (distance, index); +inf / NO_ID = empty
    A kd = pos_inf<A>();
    uint32_t ki = NO_ID;
    A kth_d = pos_inf<A>();      // key of entry k-1 (warp-uniform): the pruning bound and the admission threshold
    uint32_t kth_i = NO_ID;
    A t2 = pos_inf<A>();         // squared-domain filter for kth_d
    const uint32_t k = a.k;
    const bool has_floor = a.pass > 0;
    const A fl_d = has_floor ? a.floor_d[qid] : A(0);
    const uint32_t fl_i = has_floor ? a.floor_i[qid] : 0u;
    auto insert = [&](A cd, uint32_t ci) {   // warp-uniform candidate
        if (has_floor && !(cd > fl_d || (cd == fl_d && ci > fl_i))) return;   // already reported by an earlier pass
        const bool less = kd < cd || (kd == cd && ki < ci);
        const uint32_t pos = __popc(__ballot_sync(full, less));   // held entries smaller than the candidate: a prefix
        if (pos >= k) return;
        const A ud = __shfl_up_sync(full, kd, 1);
        const uint32_t ui = __shfl_up_sync(full, ki, 1);
        if ((uint32_t)lane > pos) { kd = ud; ki = ui; }
        else if ((uint32_t)lane == pos) { kd = cd; ki = ci; }
        kth_d = __shfl_sync(full, kd, (int)k - 1);
        kth_i = __shfl_sync(full, ki, (int)k - 1);
        t2 = kth_i == NO_ID ? pos_inf<A>() : thresh2(kth_d);
    };
    unsigned long long pairs = 0, visits = 0;
    uint32_t stack[MAX_STACK];
    A lbs[MAX_STACK];
    int sp = 0;
    stack[0] = 0; lbs[0] = -pos_inf<A>(); sp = 1;
    while (sp) {
        --sp;
        const uint32_t node = stack[sp];
        if (lbs[sp] > kth_d) continue;   // the bound has tightened since this node was pushed
        ++visits;
        if (node >= t.n_internal) {
            const uint32_t b = node - t.n_internal;
            const uint32_t lo = __ldg(t.bucket_lo + b), hi = __ldg(t.bucket_hi + b);
            pairs += hi - lo;
            for (uint32_t base = lo; base < hi; base += 32) {
                const uint32_t p = base + lane;
                A acc = pos_inf<A>();
                if (p < hi) acc = dist2_to(t.pts + (size_t)p * DV);
                unsigned mask = __ballot_sync(full, acc <= t2);
                if (!mask) continue;
                A dd = A(0);
                uint32_t id = NO_ID;
                if ((mask >> lane) & 1u) { dd = xsqrt(acc); id = __ldg(t.ids + p); }
                while (mask) {
                    const int src = __ffs(mask) - 1;
                    mask &= mask - 1;
                    const A cd = __shfl_sync(full, dd, src);
                    const uint32_t ci = __shfl_sync(full, id, src);
                    if (cd < kth_d || (cd == kth_d && ci < kth_i)) insert(cd, ci);
                }
            }
        } else {
            // lanes 0 and 1 take one child each
            const uint32_t c = 2 * node + 1 + (uint32_t)(lane & 1);
            const A R = __ldg(t.radii + c);
            A lb = pos_inf<A>();
            if (lane < 2 && !(R < A(0))) {
                const A cd = xsqrt(dist2_to(t.centers + (size_t)c * DV));
                lb = xsub(xsub(cd, R), xmul(t.slack, xadd(cd, R)));
            }
            const A lb1 = __shfl_sync(full, lb, 0), lb2 = __shfl_sync(full, lb, 1);
            const uint32_t c1 = 2 * node + 1, c2 = c1 + 1;
            const bool n1 = !(lb1 > kth_d) && lb1 < pos_inf<A>(), n2 = !(lb2 > kth_d) && lb2 < pos_inf<A>();
            // nearer child first (:232-236): it is pushed last
            if (lb1 < lb2) {
                if (n2) { stack[sp] = c2; lbs[sp] = lb2; ++sp; }
                if (n1) { stack[sp] = c1; lbs[sp] = lb1; ++sp; }
            } else {
                if (n1) { stack[sp] = c1; lbs[sp] = lb1; ++sp; }
                if (n2) { stack[sp] = c2; lbs[sp] = lb2; ++sp; }
            }
        }
    }
    const size_t orow = a.row_map ? a.row_map[qid] : qid;
    if ((uint32_t)lane < k) {
        a.out_d[orow * a.out_stride + a.out_off + lane] = kd;
        a.out_i[orow * a.out_stride + a.out_off + lane] = ki == NO_ID ? ~0ull : (uint64_t)ki;
    }
    if (a.floor_d && (uint32_t)lane == k - 1) { a.floor_d[qid] = kd; a.floor_i[qid] = ki; }
    if (a.counters && lane == 0) { atomicAdd(&a.counters[0], pairs); atomicAdd(&a.counters[1], visits); }
}

// ---- k-way merge of sorted (distance, index) lists: split scans of one GPU, or the gathered
// per-shard lists of several GPUs (K7 in SURVEY.md 2): merge_lists() below.  This kernel is its
// single-list case, one thread per query. ---------------
constexpr int MAX_LISTS = 256;
template <typename A, typename I>
__global__ void merge_lists_kernel(const A* __restrict__ in_d, const I* __restrict__ in_i, uint32_t n_lists,
                                   uint32_t nq, uint32_t k, uint64_t* __restrict__ out_i, A* __restrict__ out_d,
                                   uint32_t out_stride, uint32_t out_off, A* floor_d, uint32_t* floor_i,
                                   const uint32_t* __restrict__ row_map = nullptr) {
    const uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= nq) return;
    const size_t orow = row_map ? row_map[q] : q;  // self-query: results go to the original row of stored point q
    const I none = (I)~(I)0;
    A last_d = pos_inf<A>();
    uint64_t last_i = ~0ull;
    (void)n_lists;   // one list per query: copy (and widen the indices) to the output rows
    for (uint32_t i = 0; i < k; ++i) {
        const A d = in_d[(size_t)q * k + i];
        const I id = in_i[(size_t)q * k + i];
        out_d[orow * out_stride + out_off + i] = d;
        out_i[orow * out_stride + out_off + i] = id == none ? ~0ull : (uint64_t)id;
        last_d = d; last_i = id == none ? ~0ull : (uint64_t)id;
    }
    if (floor_d && k > 0) { floor_d[q] = last_d; floor_i[q] = last_i == ~0ull ? NO_ID : (uint32_t)last_i; }
}

// Several lists: one WARP per query.  Lane l keeps the heads of lists l, l + 32, ... (at most MAX_LISTS / 32) in
// registers; every output slot is one lane-local minimum, one five-step warp arg-min on (distance, index) and one reload
// by the winning lane -- no per-thread head array in local memory, O(k (n_lists / 32 + 5)) steps per query.
template <typename A, typename I>
__global__ void merge_lists_warp_kernel(const A* __restrict__ in_d, const I* __restrict__ in_i, uint32_t n_lists, uint32_t nq, uint32_t k,
                                        uint64_t* __restrict__ out_i, A* __restrict__ out_d, uint32_t out_stride, uint32_t out_off,
                                        A* floor_d, uint32_t* floor_i, const uint32_t* __restrict__ row_map) {
    constexpr int PER = MAX_LISTS / 32;
    const int lane = threadIdx.x & 31;
    const uint32_t q = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (q >= nq) return;
    const size_t orow = row_map ? row_map[q] : q;
    const I none = (I)~(I)0;
    const unsigned full = 0xffffffffu;
    uint32_t head[PER];
    A hd[PER];
    uint64_t hi[PER];
    auto load = [&](int s_, uint32_t h, A& d, uint64_t& id) {
        const uint32_t l = (uint32_t)lane + 32u * (uint32_t)s_;
        d = pos_inf<A>(); id = ~0ull;   // exhausted (or absent) list: never wins against a real entry
        if (l < n_lists && h < k) {
            const size_t at = ((size_t)l * nq + q) * k + h;
            const I v = in_i[at];
            if (v != none) { d = in_d[at]; id = (uint64_t)v; }
        }
    };
#pragma unroll
    for (int s_ = 0; s_ < PER; ++s_) { head[s_] = 0; load(s_, 0, hd[s_], hi[s_]); }
    A last_d = pos_inf<A>();
    uint64_t last_i = ~0ull;
    for (uint32_t i = 0; i < k; ++i) {
        A bd = hd[0];
        uint64_t bi = hi[0];
        int bs = 0;
#pragma unroll
        for (int s_ = 1; s_ < PER; ++s_)
            if (hd[s_] < bd || (hd[s_] == bd && hi[s_] < bi)) { bd = hd[s_]; bi = hi[s_]; bs = s_; }
        A wd = bd;
        uint64_t wi = bi;
        int wl = lane;
#pragma unroll
        for (int o = 16; o; o >>= 1) {
            const A od = __shfl_xor_sync(full, wd, o);
            const uint64_t oi = __shfl_xor_sync(full, wi, o);
            const int ol = __shfl_xor_sync(full, wl, o);
            if (od < wd || (od == wd && (oi < wi || (oi == wi && ol < wl)))) { wd = od; wi = oi; wl = ol; }
        }
        if (lane == wl && wi != ~0ull) {
#pragma unroll
            for (int s_ = 0; s_ < PER; ++s_)
                if (s_ == bs) { ++head[s_]; load(s_, head[s_], hd[s_], hi[s_]); }
        }
        if (lane == 0) {
            out_d[orow * out_stride + out_off + i] = wd;
            out_i[orow * out_stride + out_off + i] = wi;
        }
        last_d = wd; last_i = wi;
    }
    if (lane == 0 && floor_d && k > 0) { floor_d[q] = last_d; floor_i[q] = last_i == ~0ull ? NO_ID : (uint32_t)last_i; }
}
// one list: the copy / row-map kernel above, a thread per query; several: a warp per query
template <typename A, typename I>
inline cudaError_t merge_lists(cudaStream_t st, const A* in_d, const I* in_i, uint32_t n_lists, uint32_t nq, uint32_t k, uint64_t* out_i,
                               A* out_d, uint32_t out_stride, uint32_t out_off, A* floor_d, uint32_t* floor_i, const uint32_t* row_map = nullptr) {
    if (nq == 0) return cudaSuccess;
    if (n_lists <= 1)
        merge_lists_kernel<A, I><<<(nq + 127) / 128, 128, 0, st>>>(in_d, in_i, n_lists, nq, k, out_i, out_d, out_stride, out_off, floor_d, floor_i, row_map);
    else
        merge_lists_warp_kernel<A, I><<<(nq + 7) / 8, 256, 0, st>>>(in_d, in_i, n_lists, nq, k, out_i, out_d, out_stride, out_off, floor_d, floor_i, row_map);
    return cudaGetLastError();
}

// k > n: columns [k_eff, k) of every output row are (UINT64_MAX, +inf) -- the reference returns only n results
// (the heap never fills, src/ball_tree.rs:219-221); the fixed-shape batched output pads instead of scanning again
template <typename A>
__global__ void pad_rows_kernel(uint64_t* __restrict__ out_i, A* __restrict__ out_d, uint32_t nq, uint32_t k, uint32_t k_eff) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t w = k - k_eff;
    if (i >= (size_t)nq * w) return;
    const size_t at = (i / w) * k + k_eff + (i % w);
    out_i[at] = ~0ull;
    out_d[at] = pos_inf<A>();
}

// ---- exchange format of the sharded k-NN (f32): one 64-bit key per entry, (distance bits << 32) | index.  Distances
// are non-negative, so unsigned order of the keys is the (distance, index) order; an empty slot (+inf, NO_ID) is the
// largest key.  8 bytes per entry cross NVLink instead of 12. ----------------------------------------------------------
__global__ void pack_lists_kernel(const uint64_t* __restrict__ idx, const float* __restrict__ dist, size_t count,
                                  unsigned long long* __restrict__ out) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    const uint64_t id = idx[i];
    out[i] = ((unsigned long long)__float_as_uint(dist[i]) << 32) | (id == ~0ull ? (unsigned long long)NO_ID : (id & 0xffffffffull));
}
// k-way merge of n_lists sorted packed lists per query (K7 of SURVEY.md 2 after the exchange); lists[l * list_stride + q * k + i]
__global__ void merge_packed_kernel(const unsigned long long* __restrict__ lists, uint32_t n_lists, size_t list_stride, uint32_t nq,
                                    uint32_t k, uint64_t* __restrict__ out_i, float* __restrict__ out_d) {
    const uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= nq) return;
    uint8_t head[64];
    for (uint32_t l = 0; l < n_lists; ++l) head[l] = 0;
    for (uint32_t i = 0; i < k; ++i) {
        unsigned long long best = ~0ull;
        int bl = -1;
        for (uint32_t l = 0; l < n_lists; ++l) {
            if (head[l] >= k) continue;
            const unsigned long long key = lists[(size_t)l * list_stride + (size_t)q * k + head[l]];
            if (bl < 0 || key < best) { best = key; bl = (int)l; }
        }
        if (bl >= 0) ++head[bl];
        const uint32_t id = (uint32_t)best;
        out_d[(size_t)q * k + i] = __uint_as_float((uint32_t)(best >> 32));
        out_i[(size_t)q * k + i] = (bl < 0 || id == NO_ID) ? ~0ull : (uint64_t)id;
    }
}

// The same merge with the lists read where they were produced: lists[l] is the packed list buffer of rank l -- for l != this
// rank a PEER pointer, so the loads cross NVLink inside the merge kernel and no collective runs at all (one process driving
// several GPUs, pn_multi_*).  Rows [row_off, row_off + nq) of every rank's chunk buffer are merged.
__global__ void merge_packed_peer_kernel(const unsigned long long* const* __restrict__ lists, uint32_t n_lists, size_t row_off, uint32_t nq,
                                         uint32_t k, uint64_t* __restrict__ out_i, float* __restrict__ out_d) {
    const uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= nq) return;
    uint8_t head[64];
    for (uint32_t l = 0; l < n_lists; ++l) head[l] = 0;
    for (uint32_t i = 0; i < k; ++i) {
        unsigned long long best = ~0ull;
        int bl = -1;
        for (uint32_t l = 0; l < n_lists; ++l) {
            if (head[l] >= k) continue;
            const unsigned long long key = lists[l][(row_off + q) * k + head[l]];
            if (bl < 0 || key < best) { best = key; bl = (int)l; }
        }
        if (bl >= 0) ++head[bl];
        const uint32_t id = (uint32_t)best;
        out_d[(size_t)q * k + i] = __uint_as_float((uint32_t)(best >> 32));
        out_i[(size_t)q * k + i] = (bl < 0 || id == NO_ID) ? ~0ull : (uint64_t)id;
    }
}

// ids[i] = map[ids[i]]: the companion ball tree of a vantage-point handle is built over that handle's stored rows
__global__ void translate_ids_kernel(uint32_t* __restrict__ ids, const uint32_t* __restrict__ map, uint32_t n) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) ids[i] = map[ids[i]];
}

// ---- query staging ----------------------------------------------------------------------------
template <typename A>
__global__ void pad_queries_kernel(const A* __restrict__ q, size_t q_stride, uint32_t nq, uint32_t d, uint32_t dpad,
                                   A* __restrict__ out) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)nq * dpad) return;
    const uint32_t r = (uint32_t)(i / dpad), c = (uint32_t)(i % dpad);
    out[i] = c < d ? q[(size_t)r * q_stride + c] : A(0);
}

// home bucket of each query: greedy descent (nearer centroid / near-far side of mu).  Only used
// to sort queries so that the 128 queries of a tile visit the same buckets.
template <typename A>
__global__ void home_bucket_kernel(const DevTree<A> t, const typename VT<A>::V* __restrict__ q, uint32_t nq,
                                   uint32_t* __restrict__ home, uint32_t* __restrict__ hist) {
    using V = typename VT<A>::V;
    const uint32_t qi = blockIdx.x * blockDim.x + threadIdx.x;
    if (qi >= nq) return;
    const V* qr = q + (size_t)qi * t.dv;
    auto dist_to = [&](const V* row) {
        A acc = A(0);
        for (uint32_t jc = 0; jc < t.dv; ++jc) acc = fold(acc, qr[jc], __ldg(row + jc));
        return acc;
    };
    uint32_t node = 0;
    while (node < t.n_internal) {
        const uint32_t c1 = 2 * node + 1, c2 = c1 + 1;
        if (t.kind == 0) {
            const A R1 = t.radii[c1], R2 = t.radii[c2];
            if (R1 < A(0)) { node = c2; continue; }
            if (R2 < A(0)) { node = c1; continue; }
            if (t.plane_w) {
                // the side of the cut the points themselves were sent to (the nearer centroid disagrees with the median cut
                // for a few per cent of the queries, and a query in the wrong bucket gets a useless seed)
                const A* w = t.plane_w + (size_t)node * t.dpad;
                const A* qs = reinterpret_cast<const A*>(qr);
                A key = A(0);
                for (uint32_t j = 0; j < t.dpad; ++j) key += qs[j] * __ldg(w + j);
                node = key < t.plane_t[node] ? c1 : c2;
                continue;
            }
            node = dist_to(t.centers + (size_t)c1 * t.dv) <= dist_to(t.centers + (size_t)c2 * t.dv) ? c1 : c2;
        } else {
            const A mu = t.radii[node];
            node = xsqrt(dist_to(t.centers + (size_t)node * t.dv)) < mu ? c1 : c2;
        }
    }
    const uint32_t b = node - t.n_internal;
    home[qi] = b;
    atomicAdd(&hist[b], 1u);
}

// exclusive scan of n uint32 counters by a single block (n <= a few million)
__global__ void exclusive_scan_kernel(const uint32_t* __restrict__ in, uint32_t* __restrict__ out, uint32_t n) {
    __shared__ uint32_t sums[1024];
    const uint32_t tid = threadIdx.x, nt = blockDim.x;
    const uint32_t chunk = (n + nt - 1) / nt;
    const uint32_t b = min(n, tid * chunk), e = min(n, b + chunk);
    uint32_t s = 0;
    for (uint32_t i = b; i < e; ++i) s += in[i];
    sums[tid] = s;
    __syncthreads();
    if (tid == 0) {
        uint32_t run = 0;
        for (uint32_t i = 0; i < nt; ++i) { uint32_t v = sums[i]; sums[i] = run; run += v; }
    }
    __syncthreads();
    uint32_t run = sums[tid];
    for (uint32_t i = b; i < e; ++i) { uint32_t v = in[i]; out[i] = run; run += v; }
}

__global__ void scatter_order_kernel(const uint32_t* __restrict__ home, uint32_t* __restrict__ cursor, uint32_t nq,
                                     uint32_t* __restrict__ qorder) {
    const uint32_t qi = blockIdx.x * blockDim.x + threadIdx.x;
    if (qi >= nq) return;
    const uint32_t pos = atomicAdd(&cursor[home[qi]], 1u);
    qorder[pos] = qi;
}

// ---- radius search: one warp per query, lanes over the points of a bucket, hits compacted with
// __ballot_sync + popc prefix (neighbors_within_radius_in_subtree, src/ball_tree.rs:250-294).
// Contract (SURVEY S6): index i is reported iff the bit-exact distance is < r (strict, :277).
// A node is skipped when its conservative lower bound is >= r and taken whole, without per-point
// tests (:271-273), when its conservative upper bound is < r.  Pass 1 (out == null) counts,
// pass 2 writes at offsets[q]. ---------------------------------------------------------------
// Single traversal for the common case: MODE 0 writes the first RADIUS_CAP hits of every query into its slab
// (slab[qi * RADIUS_CAP + ..]) and the full count into counts[]; compact_hits_kernel then moves the slabs to their CSR
// positions and lists the queries whose count exceeds the slab, and only those are traversed again (MODE 1: fill at
// offsets[qi], queries taken from qlist[0 .. *n_list)).
constexpr uint32_t RADIUS_CAP = 64;
template <typename A, int MODE>
__global__ void radius_kernel(const DevTree<A> t, const typename VT<A>::V* __restrict__ q, uint32_t nq, A r,
                              uint32_t* __restrict__ counts, const uint64_t* __restrict__ offsets,
                              uint32_t* __restrict__ out, unsigned long long* counters,
                              const uint32_t* __restrict__ qlist = nullptr, const uint32_t* __restrict__ n_list = nullptr) {
    using V = typename VT<A>::V;
    const unsigned full = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const uint32_t warps_per_block = blockDim.x >> 5;
    const uint32_t w = blockIdx.x * warps_per_block + (threadIdx.x >> 5);
    if (w >= nq) return;
    uint32_t qi = w;
    if (MODE == 1) {
        if (w >= *n_list) return;
        qi = qlist[w];
    }
    const uint32_t cap = MODE == 0 ? RADIUS_CAP : 0xffffffffu;  // entries this pass may write
    const V* qr = q + (size_t)qi * t.dv;
    auto dist_to = [&](const V* row) {
        A acc = A(0);
        for (uint32_t jc = 0; jc < t.dv; ++jc) acc = fold(acc, __ldg(qr + jc), __ldg(row + jc));
        return xsqrt(acc);
    };
    const uint64_t base = MODE == 0 ? (uint64_t)qi * RADIUS_CAP : offsets[qi];
    uint32_t count = 0;
    unsigned long long pairs = 0;
    uint32_t stack[MAX_STACK];
    int sp = 0;
    stack[sp++] = 0;
    while (sp) {
        const uint32_t node = stack[--sp];
        const A R = t.radii[node];
        if (R < A(0)) continue;
        const A cd = dist_to(t.centers + (size_t)node * t.dv);  // warp-uniform
        const A s = xmul(t.slack, xadd(cd, R));
        const A lb = xsub(xsub(cd, R), s), ub = xadd(xadd(cd, R), s);
        if (lb >= r) continue;
        // leaf-bucket span of this node in the implicit complete tree
        uint32_t first = node, last = node;
        while (first < t.n_internal) { first = 2 * first + 1; last = 2 * last + 2; }
        const uint32_t lo = t.bucket_lo[first - t.n_internal], hi = t.bucket_hi[last - t.n_internal];
        if (ub < r) {  // whole node inside the ball
            for (uint32_t p = lo + lane; p < hi && count + (p - lo) < cap; p += 32) out[base + count + (p - lo)] = t.ids[p];
            count += hi - lo;
        } else if (node >= t.n_internal) {
            for (uint32_t p0 = lo; p0 < hi; p0 += 32) {
                const uint32_t p = p0 + lane;
                bool hit = false;
                if (p < hi) hit = dist_to(t.pts + (size_t)p * t.dv) < r;
                const unsigned m = __ballot_sync(full, hit);
                const uint32_t pos = count + __popc(m & ((1u << lane) - 1u));
                if (hit && pos < cap) out[base + pos] = t.ids[p];
                count += __popc(m);
            }
            pairs += hi - lo;
        } else {
            stack[sp++] = 2 * node + 1;  // :284-285
            stack[sp++] = 2 * node + 2;
        }
    }
    if (MODE == 0 && lane == 0) counts[qi] = count;
    if (counters && lane == 0) atomicAdd(&counters[0], pairs);
}

// slabs -> CSR: one warp per query copies its (at most RADIUS_CAP) hits to offsets[qi]; queries that overflowed their
// slab are appended to qlist for the second traversal
__global__ void compact_hits_kernel(const uint32_t* __restrict__ slab, const uint32_t* __restrict__ counts, const uint64_t* __restrict__ offsets,
                                    uint32_t nq, uint32_t* __restrict__ hits, uint32_t* __restrict__ qlist, uint32_t* __restrict__ n_list) {
    const int lane = threadIdx.x & 31;
    const uint32_t qi = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (qi >= nq) return;
    const uint32_t c = counts[qi];
    if (c > RADIUS_CAP) {
        if (lane == 0) qlist[atomicAdd(n_list, 1u)] = qi;
        return;
    }
    const uint64_t o = offsets[qi];
    for (uint32_t i = lane; i < c; i += 32) hits[o + i] = slab[(uint64_t)qi * RADIUS_CAP + i];
}

// u32 counts -> u64 exclusive offsets, offsets[n] = total.  Two launches over blocks of SCAN_BLOCK counts: the sums of the
// blocks, then every block adds the sums of the blocks before it (at most a few hundred values) to its own scan.
constexpr uint32_t SCAN_BLOCK = 4096;   // 1024 threads x 4 counts
__global__ void scan_sums_kernel(const uint32_t* __restrict__ counts, uint32_t n, unsigned long long* __restrict__ sums) {
    __shared__ unsigned long long ws[32];
    const uint32_t i0 = blockIdx.x * SCAN_BLOCK + threadIdx.x * 4;
    unsigned long long s = 0;
    if (i0 + 3 < n) {
        const uint4 v = *reinterpret_cast<const uint4*>(counts + i0);
        s = (unsigned long long)v.x + v.y + v.z + v.w;
    } else {
        for (uint32_t i = i0; i < n && i < i0 + 4; ++i) s += counts[i];
    }
    for (int o = 16; o; o >>= 1) s += __shfl_down_sync(0xffffffffu, s, o);
    if ((threadIdx.x & 31) == 0) ws[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x < 32) {
        s = ws[threadIdx.x];
        for (int o = 16; o; o >>= 1) s += __shfl_down_sync(0xffffffffu, s, o);
        if (threadIdx.x == 0) sums[blockIdx.x] = s;
    }
}
__global__ void offsets_scan_kernel(const uint32_t* __restrict__ counts, const unsigned long long* __restrict__ sums,
                                    uint64_t* __restrict__ offsets, uint32_t n) {
    __shared__ unsigned long long ws[33];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    // sum of the blocks before this one
    unsigned long long base = 0;
    for (uint32_t b = threadIdx.x; b < blockIdx.x; b += blockDim.x) base += sums[b];
    for (int o = 16; o; o >>= 1) base += __shfl_down_sync(0xffffffffu, base, o);
    if (lane == 0) ws[w] = base;
    __syncthreads();
    if (threadIdx.x < 32) {
        base = ws[threadIdx.x];
        for (int o = 16; o; o >>= 1) base += __shfl_down_sync(0xffffffffu, base, o);
        if (threadIdx.x == 0) ws[32] = base;
    }
    __syncthreads();
    base = ws[32];
    __syncthreads();
    const uint32_t i0 = blockIdx.x * SCAN_BLOCK + threadIdx.x * 4;
    uint32_t v[4] = {0, 0, 0, 0};
    if (i0 + 3 < n) {
        const uint4 t = *reinterpret_cast<const uint4*>(counts + i0);
        v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
    } else {
        for (uint32_t i = 0; i < 4 && i0 + i < n; ++i) v[i] = counts[i0 + i];
    }
    const unsigned long long mine = (unsigned long long)v[0] + v[1] + v[2] + v[3];
    unsigned long long inc = mine;   // inclusive scan over the warp
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned long long t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += t;
    }
    if (lane == 31) ws[w] = inc;
    __syncthreads();
    if (threadIdx.x < 32) {
        unsigned long long x = ws[threadIdx.x], xi = x;
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned long long t = __shfl_up_sync(0xffffffffu, xi, o);
            if (lane >= o) xi += t;
        }
        ws[threadIdx.x] = xi - x;   // exclusive over the warps
    }
    __syncthreads();
    unsigned long long run = base + ws[w] + inc - mine;
    for (uint32_t i = 0; i < 4 && i0 + i < n; ++i) { offsets[i0 + i] = run; run += v[i]; }
    if (i0 < n && i0 + 4 >= n) offsets[n] = run;   // the thread holding the last count
    if (n == 0 && blockIdx.x == 0 && threadIdx.x == 0) offsets[0] = 0;
}

// add to every entry of a u64 offset array: out[i] = in[i] - sub + add (chunk-local CSR offsets -> batch offsets, pulled
// offsets -> positions in the concatenation of the pulled hit lists).  in == out is allowed.
__global__ void rebase_offsets_kernel(const uint64_t* in, size_t n, uint64_t sub, uint64_t add, uint64_t* out) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = in[i] - sub + add;
}

// ---- merge of n_lists CSR radius results over the same nq queries (per-shard hit lists of a point set sharded by
// subtree).  offsets[l * (nq + 1) + q] are absolute positions into one indices array; list l holds the entries
// [offsets[l][0], offsets[l][nq]) and its segment of query q, [offsets[l][q], offsets[l][q + 1]), is non-decreasing.
// Segment lengths per query, u32, for scan_sums_kernel + offsets_scan_kernel (a decreasing pair counts as empty; a sum
// beyond u32 saturates, and merge_radius_lists_kernel then drops what no longer fits its row).
__global__ void merge_radius_counts_kernel(const uint64_t* __restrict__ offsets, uint32_t n_lists, uint32_t nq,
                                           uint32_t* __restrict__ counts) {
    const uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= nq) return;
    unsigned long long c = 0;
    for (uint32_t l = 0; l < n_lists; ++l) {
        const uint64_t a = offsets[(size_t)l * ((size_t)nq + 1) + q], b = offsets[(size_t)l * ((size_t)nq + 1) + q + 1];
        c += b > a ? b - a : 0;
    }
    counts[q] = (uint32_t)min(c, 0xffffffffull);
}

// first position in [lo, hi) whose value is > v (UPPER) or >= v (!UPPER)
template <bool UPPER, typename I>
__device__ __forceinline__ uint64_t csr_bound(const I* __restrict__ v, uint64_t lo, uint64_t hi, I x) {
    while (lo < hi) {
        const uint64_t mid = lo + (hi - lo) / 2;
        const I y = v[mid];
        if (UPPER ? y <= x : y < x) lo = mid + 1; else hi = mid;
    }
    return lo;
}

// Merge by rank, one thread per input element, no sort and no per-query work split: element j of list s's segment of
// query q (value v) goes to out_offsets[q] + j + (entries <= v in the segments of q of lists before s) + (entries < v in
// those of lists after s).  That is a stable merge: equal values from different lists are all kept, in list order, so a
// query with millions of hits costs no more than as many queries with few.  The grid strides over the n_lists entries
// counted in the list lengths (offsets[l][nq] - offsets[l][0]); every block rebuilds their prefix in shared memory, so the
// host needs to know neither the total nor any offset.  Bounds: an element is read only from its list's range
// [offsets[s][0], offsets[s][nq]), written only when its query was found (offsets[s][q] <= p < offsets[s][q + 1]), and
// only to a position inside [out_offsets[q], out_offsets[q + 1]) that is also below the sum of the list lengths (the
// capacity of out_indices: with offsets that decrease, the counts above can add up to more) -- indices that are not sorted
// or offsets that are not monotone give a wrong result, never an out-of-bounds write.
template <typename I>
__global__ void __launch_bounds__(256) merge_radius_lists_kernel(const uint64_t* __restrict__ offsets, const I* __restrict__ indices,
                                                                 uint32_t n_lists, uint32_t nq, const uint64_t* __restrict__ out_offsets,
                                                                 I* __restrict__ out_indices) {
    __shared__ unsigned long long start[MAX_LISTS + 1];   // start[l]: first element of list l in the grid's numbering
    if (threadIdx.x == 0) {
        unsigned long long s = 0;
        for (uint32_t l = 0; l < n_lists; ++l) {
            start[l] = s;
            const uint64_t a = offsets[(size_t)l * ((size_t)nq + 1)], b = offsets[(size_t)l * ((size_t)nq + 1) + nq];
            s += b > a ? b - a : 0;
        }
        start[n_lists] = s;
    }
    __syncthreads();
    const unsigned long long total = start[n_lists];
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (unsigned long long)gridDim.x * blockDim.x) {
        uint32_t lo = 0, hi = n_lists;   // the list: last l with start[l] <= i (empty lists share their start with the next)
        while (hi - lo > 1) {
            const uint32_t mid = (lo + hi) / 2;
            if (start[mid] <= i) lo = mid; else hi = mid;
        }
        const uint32_t s = lo;
        const uint64_t* os = offsets + (size_t)s * ((size_t)nq + 1);
        const uint64_t p = os[0] + (i - start[s]);
        // the query: last q with os[q] <= p
        uint32_t qa = 0, qb = nq;
        while (qb - qa > 1) {
            const uint32_t mid = qa + (qb - qa) / 2;
            if (os[mid] <= p) qa = mid; else qb = mid;
        }
        const uint32_t q = qa;
        if (!(os[q] <= p && p < os[q + 1])) continue;
        const I v = indices[p];
        uint64_t pos = out_offsets[q] + (p - os[q]);
        for (uint32_t l = 0; l < n_lists; ++l) {
            if (l == s) continue;
            const uint64_t a = offsets[(size_t)l * ((size_t)nq + 1) + q], b = offsets[(size_t)l * ((size_t)nq + 1) + q + 1];
            if (b <= a) continue;
            pos += (l < s ? csr_bound<true>(indices, a, b, v) : csr_bound<false>(indices, a, b, v)) - a;
        }
        if (pos < out_offsets[q + 1] && pos < total) out_indices[pos] = v;
    }
}
// The whole merge on `st` (nq >= 1): counts, the offsets scan, the merge on `blocks` blocks.  Workspaces: counts[nq],
// sums[nq / SCAN_BLOCK + 1].
template <typename I>
inline cudaError_t merge_radius_lists(cudaStream_t st, const uint64_t* offsets, const I* indices, uint32_t n_lists, uint32_t nq,
                                      uint64_t* out_offsets, I* out_indices, uint32_t* counts, unsigned long long* sums, unsigned blocks) {
    merge_radius_counts_kernel<<<(unsigned)(((size_t)nq + 255) / 256), 256, 0, st>>>(offsets, n_lists, nq, counts);
    const unsigned sblocks = (unsigned)(((size_t)nq + SCAN_BLOCK - 1) / SCAN_BLOCK);
    scan_sums_kernel<<<sblocks, 1024, 0, st>>>(counts, nq, sums);
    offsets_scan_kernel<<<sblocks, 1024, 0, st>>>(counts, sums, out_offsets, nq);
    merge_radius_lists_kernel<I><<<blocks, 256, 0, st>>>(offsets, indices, n_lists, nq, out_offsets, out_indices);
    return cudaGetLastError();
}

// ascending sort of each query's hit list (the reference's order is unspecified DFS order and its tests sort before
// comparing, src/ball_tree.rs:667, 777): bitonic network over the segment padded to a power of two with virtual +inf
// keys.  Segments of up to SORT_WARP_MAX entries are sorted by one warp each; longer ones (large radii: whole subtrees
// included) by one 256-thread block each in a second launch, so that a few huge hit lists do not serialise on 32 lanes.
constexpr uint32_t SORT_WARP_MAX = 1024;
// all-ascending form of the network (first step of each phase mirrors, i ^ (size-1)): every compare-exchange moves the
// smaller key down, so the virtual +inf keys at >= n never move
__device__ __forceinline__ void sort_cmpx(uint32_t* v, uint32_t n, uint32_t i, uint32_t j) {
    if (j > i && j < n) {
        const uint32_t x = v[i], y = v[j];
        if (x > y) { v[i] = y; v[j] = x; }
    }
}
__global__ void segment_sort_kernel(const uint64_t* __restrict__ offsets, uint32_t* __restrict__ vals, uint32_t nq) {
    const int lane = threadIdx.x & 31;
    const uint32_t qi = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (qi >= nq) return;
    const uint64_t lo = offsets[qi];
    const uint32_t n = (uint32_t)(offsets[qi + 1] - lo);
    if (n < 2 || n > SORT_WARP_MAX) return;
    uint32_t* v = vals + lo;
    uint32_t np2 = 1;
    while (np2 < n) np2 <<= 1;
    for (uint32_t size = 2; size <= np2; size <<= 1) {
        for (uint32_t i = lane; i < np2; i += 32) sort_cmpx(v, n, i, i ^ (size - 1));
        __syncwarp();
        for (uint32_t stride = size >> 2; stride > 0; stride >>= 1) {
            for (uint32_t i = lane; i < np2; i += 32) sort_cmpx(v, n, i, i ^ stride);
            __syncwarp();
        }
    }
}
__global__ void __launch_bounds__(256) segment_sort_large_kernel(const uint64_t* __restrict__ offsets, uint32_t* __restrict__ vals, uint32_t nq) {
  for (uint32_t qi = blockIdx.x; qi < nq; qi += gridDim.x) {   // a fixed grid walks the queries; long lists are rare
    const uint64_t lo = offsets[qi];
    const uint64_t n64 = offsets[qi + 1] - lo;
    if (n64 <= SORT_WARP_MAX) continue;        // block-uniform
    const uint32_t n = (uint32_t)n64;
    uint32_t* v = vals + lo;
    uint64_t np2 = 1;
    while (np2 < n) np2 <<= 1;
    for (uint64_t size = 2; size <= np2; size <<= 1) {
        for (uint64_t i = threadIdx.x; i < np2; i += blockDim.x) sort_cmpx(v, n, (uint32_t)i, (uint32_t)(i ^ (size - 1)));
        __syncthreads();
        for (uint64_t stride = size >> 2; stride > 0; stride >>= 1) {
            for (uint64_t i = threadIdx.x; i < np2; i += blockDim.x) sort_cmpx(v, n, (uint32_t)i, (uint32_t)(i ^ stride));
            __syncthreads();
        }
    }
  }
}


// ---- distance::pairwise (reference src/distance.rs:58-74): dense symmetric n x n matrix of exact
// fold distances.  A 32 x 32 output tile per block; the two 32-row panels are staged in shared
// memory in chunks of 32 dimensions, every thread keeps its sequential sum across chunks, so the
// result is bit-identical to the reference's per-pair fold (and symmetric: (a-b)^2 == (b-a)^2). --
// `out` holds rows [row0, row0 + rows) of the matrix: the host walks the matrix in row blocks that fit a bounded buffer.
template <typename A>
__global__ void pairwise_kernel(const A* __restrict__ x, uint32_t n, uint32_t d, A* __restrict__ out, uint32_t row0, uint32_t rows) {
    __shared__ A pi[32][33], pj[32][33];
    const uint32_t i0 = row0 + blockIdx.y * 32, j0 = blockIdx.x * 32;
    const uint32_t ti = threadIdx.y, tj = threadIdx.x;
    A acc = A(0);
    for (uint32_t c0 = 0; c0 < d; c0 += 32) {
        const uint32_t c = c0 + tj;
        pi[ti][tj] = (i0 + ti < n && c < d) ? x[(size_t)(i0 + ti) * d + c] : A(0);
        pj[ti][tj] = (j0 + ti < n && c < d) ? x[(size_t)(j0 + ti) * d + c] : A(0);
        __syncthreads();
        const uint32_t lim = min(32u, d - c0);
        for (uint32_t k = 0; k < lim; ++k) {
            const A t = xsub(pi[ti][k], pj[tj][k]);
            acc = xadd(acc, xmul(t, t));
        }
        __syncthreads();
    }
    if (i0 + ti < row0 + rows && i0 + ti < n && j0 + tj < n) out[(size_t)(i0 + ti - row0) * n + (j0 + tj)] = xsqrt(acc);
}

}  // namespace petal
