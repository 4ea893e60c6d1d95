// engine.cu -- host side of libpetal_b200.so: tree handles, workspaces, launch plans, the pipelined host-buffer calls,
// the NCCL / peer-memory multi-GPU paths and the C ABI declared in include/petal_b200.h.  No CPU fallback: every query
// entry point launches the sm_100a kernels of kernels.cuh / tc_filter.cuh / tc_prune.cuh or fails with PN_CUDA; trees
// are built by flat_tree.hpp (host) or gpu_build.cu (device).
#include <sys/mman.h>

#include <chrono>
#include <condition_variable>
#include <cstdio>
#include <cstdlib>
#include <memory>
#include <atomic>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/petal_b200.h"
#include "flat_tree.hpp"
#include "comm.hpp"
#include "gpu_build.hpp"
#include "kernels.cuh"
#include "tc_filter.cuh"

namespace petal {

static thread_local std::string g_err;
static int fail(int code, const std::string& msg) {
    g_err = msg;
    return code;
}
#define CU(...)                                                                                        \
    do {                                                                                               \
        cudaError_t e_ = (__VA_ARGS__);                                                                \
        if (e_ != cudaSuccess)                                                                         \
            return fail(e_ == cudaErrorMemoryAllocation ? PN_OOM : PN_CUDA,                            \
                        std::string(#__VA_ARGS__) + ": " + cudaGetErrorString(e_));                    \
    } while (0)
#define TRY(x)                  \
    do {                        \
        int r_ = (x);           \
        if (r_ != PN_OK) return r_; \
    } while (0)

struct DeviceGuard {
    int prev = -1;
    bool ok = true;
    explicit DeviceGuard(int dev) {
        if (cudaGetDevice(&prev) != cudaSuccess) { ok = false; (void)cudaGetLastError(); return; }
        if (prev != dev && cudaSetDevice(dev) != cudaSuccess) { ok = false; (void)cudaGetLastError(); }
    }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

// A device allocation that grows on demand and is freed on the device it was made on, whichever device is current.
struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    int device = -1;
    DevBuf() = default;
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    DevBuf(DevBuf&& o) noexcept : p(o.p), cap(o.cap), device(o.device) { o.p = nullptr; o.cap = 0; }
    DevBuf& operator=(DevBuf&& o) noexcept {
        if (this != &o) {
            release();
            p = o.p; cap = o.cap; device = o.device;
            o.p = nullptr; o.cap = 0;
        }
        return *this;
    }
    ~DevBuf() { release(); }
    int ensure(size_t bytes) {
        if (bytes <= cap) return PN_OK;
        release();
        size_t want = bytes + bytes / 8 + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e != cudaSuccess) {
            (void)cudaGetLastError();
            e = cudaMalloc(&p, bytes);
            want = bytes;
        }
        if (e != cudaSuccess) { p = nullptr; return fail(PN_OOM, std::string("cudaMalloc: ") + cudaGetErrorString(e)); }
        cap = want;
        if (cudaGetDevice(&device) != cudaSuccess) (void)cudaGetLastError();
        return PN_OK;
    }
    void release() {
        if (p) {
            DeviceGuard g(device);
            cudaFree(p);
        }
        p = nullptr; cap = 0;
    }
    template <typename T> T* as() const { return reinterpret_cast<T*>(p); }
};

// A CUDA stream, event or pinned host buffer, destroyed on the device it was created on, whichever device is current.
// create() replaces what the wrapper held; on failure the wrapper is left empty.
template <typename H, cudaError_t (*Destroy)(H)>
struct CudaHandle {
    H h = nullptr;
    int device = -1;
    CudaHandle() = default;
    CudaHandle(const CudaHandle&) = delete;
    CudaHandle& operator=(const CudaHandle&) = delete;
    CudaHandle(CudaHandle&& o) noexcept : h(o.h), device(o.device) { o.h = nullptr; }
    CudaHandle& operator=(CudaHandle&& o) noexcept {
        if (this != &o) {
            reset();
            h = o.h; device = o.device;
            o.h = nullptr;
        }
        return *this;
    }
    ~CudaHandle() { reset(); }
    void reset() {
        if (h) {
            DeviceGuard g(device);
            Destroy(h);
        }
        h = nullptr;
    }
    operator H() const { return h; }

  protected:
    int created(cudaError_t e, const char* what) {
        if (e != cudaSuccess) {
            h = nullptr;
            return fail(e == cudaErrorMemoryAllocation ? PN_OOM : PN_CUDA, std::string(what) + ": " + cudaGetErrorString(e));
        }
        if (cudaGetDevice(&device) != cudaSuccess) (void)cudaGetLastError();
        return PN_OK;
    }
};
struct Stream : CudaHandle<cudaStream_t, cudaStreamDestroy> {
    int create() { reset(); return created(cudaStreamCreateWithFlags(&h, cudaStreamNonBlocking), "cudaStreamCreateWithFlags"); }
};
struct Event : CudaHandle<cudaEvent_t, cudaEventDestroy> {
    int create(unsigned flags) { reset(); return created(cudaEventCreateWithFlags(&h, flags), "cudaEventCreateWithFlags"); }
};
struct PinnedBuf : CudaHandle<void*, cudaFreeHost> {
    int create(size_t bytes) { reset(); return created(cudaHostAlloc(&h, bytes, cudaHostAllocDefault), "cudaHostAlloc"); }
    template <typename T> T* as() const { return static_cast<T*>(h); }
};
// grows `v` to at least n events created with `flags` on the current device
static int grow_events(std::vector<Event>& v, size_t n, unsigned flags) {
    while (v.size() < n) {
        Event e;
        TRY(e.create(flags));
        v.push_back(std::move(e));
    }
    return PN_OK;
}

}  // namespace petal

using namespace petal;

// State shared by the rank threads of one pn_multi query in PEER mode: every rank's packed-list buffers and events, and a
// host barrier the rank threads meet at (an event must have been RECORDED before another rank's stream can wait on it).
// Radius search uses the barrier and the r_* fields.
struct PeerShared {
    int n = 0;
    size_t chunk = 0, n_chunks = 0;                           // the chunking of this query (the same on every rank)
    std::vector<const unsigned long long*> pack;              // [rank] packed lists of ALL queries of this call
    std::vector<std::vector<Event>> ev_scan;                  // [rank][chunk]: lists of that chunk are packed
    // radius search: [rank] CSR of the rank's shard over all queries (BY_SUBTREE), its offsets at the W + 1 slice
    // boundaries, the hits of the rank's slice; the single result, allocated by rank 0 once every slice total is known
    std::vector<const uint64_t*> r_offs;
    std::vector<const uint32_t*> r_hits;
    std::vector<int> r_dev;
    std::vector<std::vector<uint64_t>> r_bound;
    std::vector<uint64_t> r_total;
    uint64_t* r_out_offs = nullptr;
    uint64_t* r_out_hits = nullptr;
    std::mutex mu;
    std::condition_variable cv;
    int count = 0, gen = 0;
    bool failed = false;
    // returns false when some rank has failed (nobody waits for it any more)
    bool barrier() {
        std::unique_lock<std::mutex> lk(mu);
        if (failed) return false;
        const int g = gen;
        if (++count == n) { count = 0; ++gen; cv.notify_all(); return true; }
        cv.wait(lk, [&] { return gen != g || failed; });
        return !failed;
    }
    void fail() { std::lock_guard<std::mutex> lk(mu); failed = true; cv.notify_all(); }
    // the status of a rank that leaves because another one failed; on_every_rank reports the failure that released it
    static constexpr const char* RELEASED = "another rank failed";
    static int released() { return petal::fail(PN_CUDA, RELEASED); }
};

// The opaque handle.
struct pn_tree {
    virtual ~pn_tree() {}
    pn_tree_info info{};
    pn_counters counters{};
    std::mutex mu;
    bool host_only = false;
    virtual uint64_t device_bytes() const = 0;   // pn_tree_info::device_bytes
    virtual int session(pn_tree** out) = 0;
    virtual int knn_host(const void* q, size_t nq, size_t stride, size_t k, uint64_t* idx, void* dist) = 0;
    virtual int knn_dev(const void* q, size_t nq, size_t stride, size_t k, uint64_t* idx, void* dist,
                        cudaStream_t st, bool sync) = 0;
    virtual int radius_host(const void* q, size_t nq, size_t stride, double r, uint64_t** offs, uint64_t** idx) = 0;
    virtual int radius_dev(const void* q, size_t nq, size_t stride, double r, uint64_t* offs, uint64_t* idx, size_t capacity,
                           cudaStream_t st, bool sync) = 0;
    virtual int knn_self(size_t k, uint64_t* idx, void* dist, bool dev, cudaStream_t st, bool sync) = 0;
    virtual int layout(uint32_t* ids, uint32_t* blo, uint32_t* bhi, void* rad, void* cen, void* pts) = 0;
    virtual int knn_sharded(pn_comm* cm, const void* q, size_t nq, size_t stride, size_t k, uint32_t exchange, uint64_t* idx, void* dist,
                            cudaStream_t st, pn_shard_stats* stats) = 0;
    virtual int replicate_send(pn_comm* cm, int root) = 0;
    virtual size_t shard_chunk(size_t nq) const = 0;
    virtual int knn_sharded_peer(PeerShared& ps, int rank, int world, const void* q, size_t nq, size_t stride, size_t k, uint64_t* idx, void* dist,
                                 pn_shard_stats* stats) = 0;
    virtual int radius_multi(PeerShared& ps, int rank, int world, bool by_subtree, const void* q, size_t nq, size_t stride, double r,
                             pn_shard_stats* stats) = 0;
};

namespace petal {

#define NC(x)                                                                                                      \
    do {                                                                                                           \
        ncclResult_t r_ = (x);                                                                                     \
        if (r_ != ncclSuccess) return fail(PN_NCCL, std::string(#x) + ": " + cm->api->GetErrorString(r_));         \
    } while (0)

template <typename A>
struct DeviceTree {
    using V = typename VT<A>::V;
    FlatTree<A> ft;  // host copy of the flattened tree (point rows dropped after upload)
    int device = 0;
    uint32_t algo = PN_ALGO_AUTO;
    uint32_t prune_opt = 0;  // pn_prune
    bool gpu_built = false;  // the tree arrays were produced on the device (gpu_build.cu); host copies are fetched on demand
    DevBuf d_pts, d_ids, d_blo, d_bhi, d_centers, d_radii, d_vpids, d_plane_w, d_plane_t;
    DevTree<A> dt{};
    uint64_t bytes = 0;      // device memory of this tree's arrays (not counting `part`)
    // tensor path (f32 input only): augmented FP16 operands, see tc_filter.cuh
    DevBuf d_baug, d_center;
    bool tensor_ready = false;
    uint32_t kp = 0;       // padded K of the augmented operands (multiple of 32)
    float pmax = 0.f;      // max |s (p - center)|
    float tscale = 1.f;    // s: power of two bringing the centred coordinates into [-1, 1]
    // pruned tensor scan (tc_prune.cuh): tile balls and the build-time estimate of what pruning can do
    DevBuf d_tcen, d_trad;
    double prune_frac = 0.0;      // estimated fraction of (query group, tile) pairs that are out of reach
    double seed_candidates = 0.0; // estimated candidates per query that survive a seed threshold
    double tile_frac = 0.0;       // estimated share of tiles beyond a single query's seed
    bool prune_on = false, tiles_on = false;   // prune_on: sorted + seeded scan; tiles_on: with tile bitmaps
    // Vantage-point trees: the tensor path never used the VP bounds (a dense scan over the stored order), and the VP order
    // -- shells around vantage points -- gives tiles that no ball can bound tightly.  A VP tree with a device therefore
    // also keeps the BALL partition of the same points (built on the device) and answers tensor-path queries from it:
    // exact 1-NN does not depend on the partition; the VP arrays serve the pruned SIMT traversal (PN_ALGO_SIMT), the layout
    // accessors and trees the tensor path does not take (f64, d < 16).
    // Ball trees (and the ball partition of a VP tree) on CLUSTERED data: the reference's split -- the median of the
    // widest coordinate -- cuts through clusters, so in d >= 32 most 128-row tiles of the stored order mix fragments of
    // several clusters and no ball bounds them tightly (BASELINE config 3: 88 % of all (query group, tile) pairs stay).
    // Such a tree keeps a second ball tree over the same rows, partitioned by the TWO-MEANS rule of gpu_build.cu
    // (partition_rule 1), and answers its k-NN batches from it: exact results do not depend on the partition, the tile
    // bitmaps of tc_prune.cuh do.  two_means_partition() decides from the build-time estimates of both partitions.
    // `part` is set when the tree is built, or once later by companion(); read it with partition().
    std::shared_ptr<DeviceTree> part;
    std::mutex part_mu;           // serialises companion() builds
    uint32_t partition_rule = 0;  // gb::build_ball_tree rule of THIS tree's arrays
    static constexpr uint32_t TWO_MEANS_ORDER_LEVELS = 1;

    std::shared_ptr<DeviceTree> partition() const { return std::atomic_load(&part); }

    // ---- device-side construction (gpu_build.cu): raw rows on the device -> the same arrays upload() would have sent
    static gb::BallOut<A> alloc_tree_arrays(void* ctx, uint64_t n, const gb::TreeShape& shape) {
        DeviceTree* e = static_cast<DeviceTree*>(ctx);
        FlatTree<A>& t = e->ft;
        t.kind = 0; t.n = n;
        t.dpad = (uint32_t)((t.d + VT<A>::N - 1) / VT<A>::N * VT<A>::N);
        t.L = shape.L; t.n_internal = (1u << t.L) - 1; t.n_buckets = 1u << t.L; t.n_nodes = (1u << (t.L + 1)) - 1;
        const auto& seg = shape.seg[t.L];
        t.bucket_lo.assign(seg.begin(), seg.end() - 1);
        t.bucket_hi.assign(seg.begin() + 1, seg.end());
        t.bucket_max = 0;
        for (uint32_t b = 0; b < t.n_buckets; ++b) t.bucket_max = std::max(t.bucket_max, t.bucket_hi[b] - t.bucket_lo[b]);
        gb::BallOut<A> o{nullptr, nullptr, nullptr, nullptr};
        if (e->d_pts.ensure((size_t)n * t.dpad * sizeof(A)) != PN_OK || e->d_ids.ensure((size_t)n * 4) != PN_OK ||
            e->d_centers.ensure((size_t)t.n_nodes * t.dpad * sizeof(A)) != PN_OK || e->d_radii.ensure((size_t)t.n_nodes * sizeof(A)) != PN_OK)
            return o;
        o.pts = e->d_pts.template as<A>(); o.ids = e->d_ids.template as<uint32_t>();
        o.centers = e->d_centers.template as<A>(); o.radii = e->d_radii.template as<A>();
        if (e->partition_rule == 1 && t.n_internal &&
            e->d_plane_w.ensure((size_t)t.n_internal * t.dpad * sizeof(A)) == PN_OK && e->d_plane_t.ensure((size_t)t.n_internal * sizeof(A)) == PN_OK) {
            o.plane_w = e->d_plane_w.template as<A>(); o.plane_t = e->d_plane_t.template as<A>();
        }
        return o;
    }
    static gb::VpOut<A> alloc_vp_arrays(void* ctx, uint64_t n, const gb::VpShape& shape) {
        DeviceTree* e = static_cast<DeviceTree*>(ctx);
        FlatTree<A>& t = e->ft;
        t.kind = 1; t.n = n; t.n_total = n;
        t.dpad = (uint32_t)((t.d + VT<A>::N - 1) / VT<A>::N * VT<A>::N);
        t.L = shape.L; t.n_internal = (1u << t.L) - 1; t.n_buckets = 1u << t.L; t.n_nodes = t.n_internal;
        t.bucket_lo = shape.lo[t.L]; t.bucket_hi = shape.hi[t.L];
        t.bucket_max = 0;
        for (uint32_t b = 0; b < t.n_buckets; ++b) t.bucket_max = std::max(t.bucket_max, t.bucket_hi[b] - t.bucket_lo[b]);
        gb::VpOut<A> o{nullptr, nullptr, nullptr, nullptr, nullptr};
        const size_t nn = std::max<uint32_t>(t.n_nodes, 1);
        if (e->d_pts.ensure((size_t)n * t.dpad * sizeof(A)) != PN_OK || e->d_ids.ensure((size_t)n * 4) != PN_OK ||
            e->d_centers.ensure(nn * t.dpad * sizeof(A)) != PN_OK || e->d_radii.ensure(nn * sizeof(A)) != PN_OK || e->d_vpids.ensure(nn * 4) != PN_OK)
            return o;
        o.pts = e->d_pts.template as<A>(); o.ids = e->d_ids.template as<uint32_t>();
        o.centers = e->d_centers.template as<A>(); o.radii = e->d_radii.template as<A>(); o.vp_ids = e->d_vpids.template as<uint32_t>();
        return o;
    }
    // vantage-point tree on the device (gb::build_vp_tree): the same arrays the host VpBuilder + upload() produce
    int build_vp_on_device(const A* raw_dev, size_t n, size_t d, size_t stride, uint32_t bucket, cudaStream_t st) {
        DeviceGuard g(device);
        if (!g.ok) return fail(PN_CUDA, "no usable CUDA device (there is no CPU fallback)");
        ft.d = (uint32_t)d;
        gb::VpShape shape;
        std::string err;
        const int rc = gb::build_vp_tree<A>(raw_dev, n, (uint32_t)d, stride, bucket, shape, &DeviceTree::alloc_vp_arrays, this, st, err);
        if (rc) return fail(rc == (int)cudaErrorMemoryAllocation ? PN_OOM : PN_CUDA, "device tree build: " + err);
        gpu_built = true;
        TRY(d_blo.ensure(ft.bucket_lo.size() * 4));
        TRY(d_bhi.ensure(ft.bucket_hi.size() * 4));
        CU(cudaMemcpy(d_blo.p, ft.bucket_lo.data(), ft.bucket_lo.size() * 4, cudaMemcpyHostToDevice));
        CU(cudaMemcpy(d_bhi.p, ft.bucket_hi.data(), ft.bucket_hi.size() * 4, cudaMemcpyHostToDevice));
        bytes = d_pts.cap + d_ids.cap + d_blo.cap + d_bhi.cap + d_centers.cap + d_radii.cap + d_vpids.cap;
        fill_dev_tree();
        TRY(prepare_tensor(st));
        return PN_OK;
    }

    int build_on_device(const A* raw_dev, size_t n_all, size_t d, size_t stride, uint32_t bucket, uint32_t shard_depth, uint32_t shard_index,
                        uint32_t rule, cudaStream_t st) {
        DeviceGuard g(device);
        if (!g.ok) return fail(PN_CUDA, "no usable CUDA device (there is no CPU fallback)");
        ft.d = (uint32_t)d; ft.n_total = n_all;
        partition_rule = rule;
        gb::TreeShape shape;
        uint64_t n = 0;
        std::string err;
        // two-means partition: the rows of a bucket follow one more level of the split (a bucket is about two tiles of the
        // tensor path's point image)
        const int rc = gb::build_ball_tree<A>(raw_dev, n_all, (uint32_t)d, stride, bucket, shard_depth, shard_index, shape, &n,
                                              &DeviceTree::alloc_tree_arrays, this, st, err, rule, rule == 1 ? TWO_MEANS_ORDER_LEVELS : 0u);
        if (rc) return fail(rc == (int)cudaErrorMemoryAllocation ? PN_OOM : PN_CUDA, "device tree build: " + err);
        if (n == 0) return fail(PN_EMPTY, "shard holds no points");
        gpu_built = true;
        TRY(d_blo.ensure(ft.bucket_lo.size() * 4));
        TRY(d_bhi.ensure(ft.bucket_hi.size() * 4));
        TRY(d_vpids.ensure(16));
        CU(cudaMemcpy(d_blo.p, ft.bucket_lo.data(), ft.bucket_lo.size() * 4, cudaMemcpyHostToDevice));
        CU(cudaMemcpy(d_bhi.p, ft.bucket_hi.data(), ft.bucket_hi.size() * 4, cudaMemcpyHostToDevice));
        bytes = d_pts.cap + d_ids.cap + d_blo.cap + d_bhi.cap + d_centers.cap + d_radii.cap + d_vpids.cap + d_plane_w.cap + d_plane_t.cap;
        fill_dev_tree();
        TRY(prepare_tensor(st));
        return PN_OK;
    }

    int upload(cudaStream_t st) {
        DeviceGuard g(device);
        if (!g.ok) return fail(PN_CUDA, "no usable CUDA device (there is no CPU fallback)");
        auto up = [&](DevBuf& b, const void* src, size_t bytes) -> int {
            TRY(b.ensure(bytes ? bytes : 16));
            if (bytes) CU(cudaMemcpy(b.p, src, bytes, cudaMemcpyHostToDevice));
            return PN_OK;
        };
        TRY(up(d_pts, ft.pts.data(), ft.pts.size() * sizeof(A)));
        TRY(up(d_ids, ft.ids.data(), ft.ids.size() * 4));
        TRY(up(d_blo, ft.bucket_lo.data(), ft.bucket_lo.size() * 4));
        TRY(up(d_bhi, ft.bucket_hi.data(), ft.bucket_hi.size() * 4));
        TRY(up(d_centers, ft.centers.data(), ft.centers.size() * sizeof(A)));
        TRY(up(d_radii, ft.radii.data(), ft.radii.size() * sizeof(A)));
        TRY(up(d_vpids, ft.vp_ids.data(), ft.vp_ids.size() * 4));
        bytes = d_pts.cap + d_ids.cap + d_blo.cap + d_bhi.cap + d_centers.cap + d_radii.cap + d_vpids.cap;
        fill_dev_tree();
        TRY(prepare_tensor(st));
        std::vector<A>().swap(ft.pts);  // the device copy is the point store from here on
        return PN_OK;
    }

    void fill_dev_tree() {
        dt.pts = d_pts.as<V>(); dt.ids = d_ids.as<uint32_t>();
        dt.bucket_lo = d_blo.as<uint32_t>(); dt.bucket_hi = d_bhi.as<uint32_t>();
        dt.centers = d_centers.as<V>(); dt.radii = d_radii.as<A>(); dt.vp_ids = d_vpids.as<uint32_t>();
        dt.n = (uint32_t)ft.n; dt.d = ft.d; dt.dpad = ft.dpad; dt.dv = ft.dpad / VT<A>::N;
        dt.L = ft.L; dt.n_internal = ft.n_internal; dt.n_buckets = ft.n_buckets; dt.n_nodes = ft.n_nodes;
        dt.kind = ft.kind;
        dt.plane_w = partition_rule == 1 && d_plane_w.p && d_plane_t.p ? d_plane_w.as<A>() : nullptr;
        dt.plane_t = dt.plane_w ? d_plane_t.as<A>() : nullptr;
        const double u = sizeof(A) == 4 ? 5.9604644775390625e-08 : 1.1102230246251565e-16;
        dt.slack = (A)((2.0 * ft.d + 8.0) * u);
    }

    // the resident A operand (nkc chunks of 8 KB per 128-query subtile) must fit shared memory: Kp <= 384
    bool tensor_eligible() const { return sizeof(A) == 4 && algo != PN_ALGO_SIMT && (algo == PN_ALGO_TENSOR || ft.d >= 16) && ft.d + tc::NSLOT <= 384; }
    int prepare_tensor(cudaStream_t st) {
        if constexpr (sizeof(A) == 4) {
            if (!tensor_eligible()) return PN_OK;
            kp = (ft.d + tc::NSLOT + tc::KC - 1) / tc::KC * tc::KC;
            // centre = mean of the stored points (double accumulation), then the largest centred coordinate.  Both passes
            // run over fixed chunks of 4096 rows and combine the chunk partials in chunk order, so the result depends
            // neither on the number of host threads nor on where it is computed: on the host for host-built trees (the
            // rows are still there), on the device for device-built ones (gb::centre_and_range_f32, the same sums).
            std::vector<float> c(ft.dpad, 0.f);
            float maxabs = 0.f;
            TRY(d_center.ensure(ft.dpad * 4));
            if (gpu_built) {
                std::string err;
                if (gb::centre_and_range_f32(d_pts.as<float>(), ft.n, ft.d, ft.dpad, d_center.as<float>(), c.data(), &maxabs, st, err))
                    return fail(PN_CUDA, "tensor path set-up: " + err);
            } else {
                const size_t CH = 4096, n_ch = (ft.n + CH - 1) / CH;
                const unsigned nt = (unsigned)std::max<size_t>(1, std::min<size_t>({n_ch, 32, std::max(1u, std::thread::hardware_concurrency())}));
                auto chunks = [&](auto&& body) {  // body(chunk index), chunks dealt round-robin to nt threads
                    std::vector<std::thread> th;
                    for (unsigned w = 1; w < nt; ++w) th.emplace_back([&, w] { for (size_t c = w; c < n_ch; c += nt) body(c); });
                    for (size_t c = 0; c < n_ch; c += nt) body(c);
                    for (auto& t : th) t.join();
                };
                std::vector<double> part(n_ch * ft.dpad, 0.0);
                chunks([&](size_t c) {
                    double* m = &part[c * ft.dpad];
                    for (size_t i = c * CH, e = std::min<size_t>(ft.n, (c + 1) * CH); i < e; ++i)
                        for (uint32_t j = 0; j < ft.d; ++j) m[j] += (double)ft.pts[i * ft.dpad + j];
                });
                std::vector<double> mean(ft.dpad, 0.0);
                for (size_t ch = 0; ch < n_ch; ++ch)
                    for (uint32_t j = 0; j < ft.d; ++j) mean[j] += part[ch * ft.dpad + j];
                for (uint32_t j = 0; j < ft.d; ++j) c[j] = (float)(mean[j] / (double)ft.n);
                std::vector<float> pmaxabs(n_ch, 0.f);
                chunks([&](size_t ch) {
                    float m = 0.f;
                    for (size_t i = ch * CH, e = std::min<size_t>(ft.n, (ch + 1) * CH); i < e; ++i)
                        for (uint32_t j = 0; j < ft.d; ++j) m = std::max(m, std::fabs(ft.pts[i * ft.dpad + j] - c[j]));
                    pmaxabs[ch] = m;
                });
                for (size_t ch = 0; ch < n_ch; ++ch) maxabs = std::max(maxabs, pmaxabs[ch]);
                CU(cudaMemcpy(d_center.p, c.data(), ft.dpad * 4, cudaMemcpyHostToDevice));
            }
            int ex = 0;
            if (maxabs > 0.f && std::isfinite(maxabs)) { std::frexp(maxabs, &ex); }  // maxabs = m 2^ex, m in [0.5, 1)
            tscale = std::ldexp(1.0f, -ex);
            // data spans so small (or so large) that s or s^2 leaves the normal float range: the scaled operands would
            // hold inf/NaN and the filter would silently drop candidates -- such trees stay on the exact scan
            if (!std::isnormal(tscale) || !std::isnormal(tscale * tscale) || !std::isfinite(maxabs)) { tensor_ready = false; return PN_OK; }
            const size_t baug_bytes = (ft.n + tc::BN - 1) / tc::BN * tc::BN * (size_t)kp * 2;  // whole tiles
            TRY(d_baug.ensure(baug_bytes));
            CU(cudaMemsetAsync(d_baug.p, 0, baug_bytes, st));
            DevBuf cnt;   // device-side results of the set-up kernels
            TRY(cnt.ensure(256));
            CU(cudaMemset(cnt.p, 0, 256));
            tc::build_baug_kernel<<<(unsigned)((ft.n + 127) / 128), 128, 0, st>>>(d_pts.as<float>(), d_center.as<float>(), tscale, (uint32_t)ft.n, ft.d,
                                                                                     ft.dpad, kp, d_baug.as<__half>(), cnt.as<unsigned int>());
            CU(cudaGetLastError());
            unsigned int bits = 0;
            CU(cudaMemcpyAsync(&bits, cnt.p, 4, cudaMemcpyDeviceToHost, st));
            CU(cudaStreamSynchronize(st));
            memcpy(&pmax, &bits, 4);
            bytes += d_baug.cap;
            tensor_ready = true;
            // tile balls for the pruned scan, and the estimate that decides whether pruning is worth its set-up passes
            const uint32_t n_tiles = (uint32_t)((ft.n + tc::BN - 1) / tc::BN);
            TRY(d_tcen.ensure((size_t)n_tiles * ft.dpad * 4));
            TRY(d_trad.ensure((size_t)n_tiles * 4));
            tc::tile_balls_kernel<<<n_tiles, 128, ft.dpad * 4, st>>>(d_pts.as<float>(), (uint32_t)ft.n, ft.d, ft.dpad, d_tcen.as<float>(), d_trad.as<float>());
            CU(cudaGetLastError());
            CU(cudaMemsetAsync(cnt.p, 0, 256, st));
            const uint32_t n_samples = std::min<uint32_t>(64u, n_tiles);
            tc::prune_estimate_kernel<<<n_samples, 256, 0, st>>>(d_tcen.as<float>(), d_trad.as<float>(), n_tiles, ft.dpad, n_samples,
                                                                     cnt.as<unsigned long long>());
            CU(cudaGetLastError());
            unsigned long long est[2] = {0, 0};
            CU(cudaMemcpyAsync(est, cnt.p, 16, cudaMemcpyDeviceToHost, st));
            CU(cudaStreamSynchronize(st));
            prune_frac = est[1] ? (double)est[0] / (double)est[1] : 0.0;
            // ... and whether seeding is: candidates a query still reranks when it starts from its home-bucket seed
            {
                const uint32_t S = std::min<uint32_t>(128u, (uint32_t)ft.n), M = (uint32_t)std::min<uint64_t>(16384u, ft.n);
                std::vector<uint32_t> rows(S), bks(S);
                for (uint32_t i = 0; i < S; ++i) {
                    rows[i] = (uint32_t)(((uint64_t)i * ft.n) / S);
                    // the bucket that stores the row; vantage points sit between buckets and use the next one
                    const uint32_t b = (uint32_t)(std::upper_bound(ft.bucket_hi.begin(), ft.bucket_hi.end(), rows[i]) - ft.bucket_hi.begin());
                    bks[i] = std::min(b, ft.n_buckets - 1);
                }
                DevBuf sr, sb;
                TRY(sr.ensure(S * 4)); TRY(sb.ensure(S * 4));
                CU(cudaMemcpyAsync(sr.p, rows.data(), S * 4, cudaMemcpyHostToDevice, st));
                CU(cudaMemcpyAsync(sb.p, bks.data(), S * 4, cudaMemcpyHostToDevice, st));
                tc::seed_estimate_kernel<<<S, 256, 0, st>>>(*reinterpret_cast<DevTree<float>*>(&dt), sr.as<uint32_t>(), sb.as<uint32_t>(), M,
                                                               d_tcen.as<float>(), d_trad.as<float>(), n_tiles, cnt.as<unsigned long long>());
                CU(cudaGetLastError());
                unsigned long long se[4] = {0, 0, 0, 0};
                CU(cudaMemcpyAsync(se, (char*)cnt.p + 16, 32, cudaMemcpyDeviceToHost, st));
                CU(cudaStreamSynchronize(st));
                seed_candidates = se[1] ? (double)se[0] / (double)se[1] * (double)ft.n : (double)ft.n;
                tile_frac = se[3] ? (double)se[2] / (double)se[3] : 0.0;
            }
            // the streaming threshold alone leaves ~k ln(n/k) + 128 candidates per query (k = 10); seeding is worth its sort
            // and bucket pass when it gets within a small multiple of that
            const double stream_candidates = 10.0 * std::log(std::max(2.0, (double)ft.n / 10.0)) + 128.0;
            const bool can = ft.n_buckets > 1 && n_tiles > 4;
            // tile bitmaps: worth their pass when a single query could skip most tiles (a CTA needs the union over its queries)
            tiles_on = can && (prune_opt == PN_PRUNE_ON || (prune_opt == PN_PRUNE_AUTO && (prune_frac >= 0.25 || tile_frac >= 0.6)));
            prune_on = can && (tiles_on || (prune_opt == PN_PRUNE_AUTO && seed_candidates <= 4.0 * stream_candidates));
            bytes += d_tcen.cap + d_trad.cap;
        }
        return PN_OK;
    }

    // subtiles per CTA: 4 (one accumulator stage each) for narrow rows, where the epilogue is the bound; 2 (two
    // stages each) where the tensor pipe is; 1 when the resident A operand of two subtiles no longer fits
    int filter_subtiles(uint32_t nkc) const {
#ifdef PN_TC_PROFILE
        if (getenv("PN_TC_MT")) return atoi(getenv("PN_TC_MT"));
#endif
        // measured (scripts/mt_sweep.sh, 1M points, k = 10): d = 16: 208 -> 165 ms; d = 64: 58.0 -> 51.0 ms; d = 96 (Kp = 128,
        // the resident A operand of four subtiles would take 128 KB): 68.1 -> 65.5 ms, not worth the shallow ring
#if defined(PN_TC_PROFILE) || defined(PN_TC_EXPERIMENTS)
        // experiment (PN_TC_MT3=1): two or three chunks with at most five K steps of data (27 <= d <= 74): THREE subtiles
        // with their A operands in tensor memory (TS-form MMA, 70 instead of 86.5 cycles).  Bit-exact, and slower: the
        // one-stage subtiles are bound by the MMA -> read-out -> release chain, not by the pipe (1M x 64, 227 328
        // queries, k = 1: 32.7 -> 36.6 ms; profiles/r02_mma_rate.md)
        static const int mt3 = getenv("PN_TC_MT3") ? atoi(getenv("PN_TC_MT3")) : 0;
        if (mt3 && nkc <= 3 && ft.d + tc::NSLOT <= 80) return 3;
#endif
        return nkc <= 3 ? 4 : (nkc <= 6 ? 2 : 1);
    }
    // queries per CTA of the scan a k-NN batch on this tree runs (on the partition, when there is one)
    size_t query_tile() const {
        const auto p = partition();
        const DeviceTree& s = p ? *p : *this;
        return s.tensor_ready ? (size_t)128 * s.filter_subtiles(s.kp / tc::KC) : 512;
    }

    // A ball tree over the points of this tree, for `part`.  `rows` (n x d, row stride `stride`) are either the
    // original-order rows or this tree's stored rows (d_pts); then the new tree's ids (positions in this tree's stored
    // order) are translated to the original point indices.
    int build_partition(const A* rows, size_t stride, uint32_t bucket, uint32_t rule, cudaStream_t st, std::shared_ptr<DeviceTree>& out) const {
        auto p = std::make_shared<DeviceTree>();
        p->device = device; p->algo = algo; p->prune_opt = prune_opt;
        TRY(p->build_on_device(rows, ft.n, ft.d, stride, bucket, 0, 0, rule, st));
        if (rows == d_pts.as<A>()) {
            translate_ids_kernel<<<(unsigned)((ft.n + 255) / 256), 256, 0, st>>>(p->d_ids.template as<uint32_t>(), d_ids.as<uint32_t>(), (uint32_t)ft.n);
            CU(cudaGetLastError());
            CU(cudaStreamSynchronize(st));
        }
        p->ft.n_total = ft.n_total;
        out = std::move(p);
        return PN_OK;
    }

    // A second ball tree over this tree's stored rows, split by the two-means rule, when that pays (see `part`):
    // AUTO tries it where seeding already pays and the tile balls of the reference partition leave a single query more than
    // a tenth of the tiles, and keeps it when its own estimates turn the bitmaps on and a single query can skip at least a
    // tenth of all tiles more; PN_PARTITION_TWO_MEANS keeps it regardless.  Returns the new
    // tree in `out` (null: stay with this partition); a failure on the way only loses the speed-up.
    void two_means_partition(uint32_t partition_opt, uint32_t bucket, cudaStream_t st, std::shared_ptr<DeviceTree>& out) const {
        out.reset();
        if constexpr (sizeof(A) == 4) {
            if (partition_opt == PN_PARTITION_REFERENCE || ft.kind != 0 || !tensor_ready || ft.n != ft.n_total) return;
            const bool forced = partition_opt == PN_PARTITION_TWO_MEANS;
            // AUTO: seeding pays (clustered data), a single query could skip some tiles but not nearly all of them
            if (forced ? ft.n < 1024 : !(ft.n >= 32768 && prune_opt == PN_PRUNE_AUTO && prune_on && tile_frac >= 0.1 && tile_frac < 0.9)) return;
            DeviceGuard g(device);
            if (!g.ok) return;
            std::shared_ptr<DeviceTree> tm;
            if (build_partition(d_pts.as<A>(), ft.dpad, bucket, 1, st, tm) != PN_OK || !tm->tensor_ready) { (void)cudaGetLastError(); return; }
            if (forced || (tm->tiles_on && tm->tile_frac >= tile_frac + 0.1)) out = std::move(tm);
        }
    }

    // A vantage-point tree's ball partition of the same points (`part`).  Tensor-eligible trees get it when they are
    // created; the others on the first query the VP arrays do not serve (radius search), whichever handle of the tree asks
    // first: built once, on the device, from the stored rows.  A failed build publishes nothing.
    int companion(cudaStream_t st, std::shared_ptr<DeviceTree>& out) {
        out = partition();
        if (out) return PN_OK;
        std::lock_guard<std::mutex> lk(part_mu);
        out = partition();
        if (out) return PN_OK;
        TRY(build_partition(d_pts.as<A>(), ft.dpad, 256, 0, st, out));
        std::atomic_store(&part, out);
        return PN_OK;
    }

    // ---- replication of the flattened tree over NCCL (query sharding: build once, broadcast) ------------------------------
    struct ReplicaHeader {
        uint64_t n, n_total;
        uint32_t d, dpad, L, n_internal, n_buckets, n_nodes, bucket_max, kp;
        int32_t kind;
        uint32_t algo, tensor_ready, prune_on;
        float pmax, tscale;
    };
    std::vector<std::pair<DevBuf*, size_t>> replica_arrays() {
        std::vector<std::pair<DevBuf*, size_t>> v = {
            {&d_pts, (size_t)ft.n * ft.dpad * sizeof(A)}, {&d_ids, (size_t)ft.n * 4}, {&d_blo, (size_t)ft.n_buckets * 4}, {&d_bhi, (size_t)ft.n_buckets * 4},
            {&d_centers, (size_t)std::max<uint32_t>(ft.n_nodes, 1) * ft.dpad * sizeof(A)}, {&d_radii, (size_t)std::max<uint32_t>(ft.n_nodes, 1) * sizeof(A)},
            {&d_vpids, ft.kind == 1 ? (size_t)std::max<uint32_t>(ft.n_nodes, 1) * 4 : 16}};
        if (partition_rule == 1 && ft.n_internal) {   // (never replicated: a tree's second partition stays on its device)
            v.push_back({&d_plane_w, (size_t)ft.n_internal * ft.dpad * sizeof(A)});
            v.push_back({&d_plane_t, (size_t)ft.n_internal * sizeof(A)});
        }
        if (tensor_ready) {
            v.push_back({&d_center, (size_t)ft.dpad * 4});
            v.push_back({&d_baug, (ft.n + tc::BN - 1) / tc::BN * tc::BN * (size_t)kp * 2});
            const size_t n_tiles = (ft.n + tc::BN - 1) / tc::BN;
            v.push_back({&d_tcen, n_tiles * ft.dpad * 4});
            v.push_back({&d_trad, n_tiles * 4});
        }
        return v;
    }
    int replicate_send(pn_comm* cm, int root) {
        ReplicaHeader h{ft.n, ft.n_total, ft.d, ft.dpad, ft.L, ft.n_internal, ft.n_buckets, ft.n_nodes, ft.bucket_max, kp, ft.kind, algo,
                        tensor_ready ? 1u : 0u, (prune_on ? 1u : 0u) | (tiles_on ? 2u : 0u), pmax, tscale};
        DevBuf hb;
        TRY(hb.ensure(sizeof(h)));
        CU(cudaMemcpyAsync(hb.p, &h, sizeof(h), cudaMemcpyHostToDevice, cm->stream));
        NC(cm->api->Broadcast(hb.p, hb.p, sizeof(h), ncclUint8, root, cm->comm, cm->stream));
        for (auto& a : replica_arrays()) NC(cm->api->Broadcast(a.first->p, a.first->p, a.second, ncclUint8, root, cm->comm, cm->stream));
        CU(cudaStreamSynchronize(cm->stream));
        return PN_OK;
    }
    int replicate_recv(pn_comm* cm, int root) {
        device = cm->device;
        DeviceGuard g(device);
        if (!g.ok) return fail(PN_CUDA, "cudaSetDevice failed");
        ReplicaHeader h{};
        DevBuf hb;
        TRY(hb.ensure(sizeof(h)));
        NC(cm->api->Broadcast(hb.p, hb.p, sizeof(h), ncclUint8, root, cm->comm, cm->stream));
        CU(cudaMemcpyAsync(&h, hb.p, sizeof(h), cudaMemcpyDeviceToHost, cm->stream));
        CU(cudaStreamSynchronize(cm->stream));
        ft.n = h.n; ft.n_total = h.n_total; ft.d = h.d; ft.dpad = h.dpad; ft.L = h.L; ft.n_internal = h.n_internal; ft.n_buckets = h.n_buckets;
        ft.n_nodes = h.n_nodes; ft.bucket_max = h.bucket_max; ft.kind = h.kind; kp = h.kp; algo = h.algo; tensor_ready = h.tensor_ready != 0;
        pmax = h.pmax; tscale = h.tscale; prune_on = (h.prune_on & 1u) != 0; tiles_on = (h.prune_on & 2u) != 0;
        gpu_built = true;  // no host copies: layout() reads the device arrays
        bytes = 0;
        for (auto& a : replica_arrays()) {
            TRY(a.first->ensure(a.second));
            NC(cm->api->Broadcast(a.first->p, a.first->p, a.second, ncclUint8, root, cm->comm, cm->stream));
            bytes += a.first->cap;
        }
        CU(cudaStreamSynchronize(cm->stream));
        ft.bucket_lo.resize(ft.n_buckets); ft.bucket_hi.resize(ft.n_buckets);
        CU(cudaMemcpy(ft.bucket_lo.data(), d_blo.p, (size_t)ft.n_buckets * 4, cudaMemcpyDeviceToHost));
        CU(cudaMemcpy(ft.bucket_hi.data(), d_bhi.p, (size_t)ft.n_buckets * 4, cudaMemcpyDeviceToHost));
        if (ft.kind == 1) {
            ft.vp_ids.resize(std::max<uint32_t>(ft.n_nodes, 1));
            CU(cudaMemcpy(ft.vp_ids.data(), d_vpids.p, ft.vp_ids.size() * 4, cudaMemcpyDeviceToHost));
        }
        fill_dev_tree();
        return PN_OK;
    }
};

template <typename A>
struct Engine final : pn_tree {
    using V = typename VT<A>::V;
    // the tree this handle queries, shared with the handle's sessions (pn_tree_session) and never written after its build,
    // except that DeviceTree::companion() may publish a partition
    std::shared_ptr<DeviceTree<A>> tree;
    bool owns_tree = true;   // false for a session: device_bytes are reported by the handle that built the tree
    int n_sms = 148;
    bool last_used_tensor = false;
    bool last_pruned = false, last_tiles = false;   // the last k-NN scan was seeded / also used tile bitmaps
    static constexpr size_t PIN_BYTES = 16u << 20;

    // Members are destroyed in reverse order of declaration, so the order of the three groups below is the teardown
    // order: events and pinned staging first, then the streams, then the device buffers.
    DevBuf w_qraw, w_q, w_home, w_hist, w_cursor, w_order, w_part_d, w_part_i, w_floor_d, w_floor_i,
        w_counters, w_out_i, w_out_d, w_counts, w_offsets, w_hits;
    // host-buffer calls are software-pipelined over chunks of queries: H2D of chunk i+1 and D2H of chunk i-1 run on their own
    // streams under the kernels of chunk i (two sets of raw-query / result buffers)
    DevBuf w_qraw2[2], w_oi2[2], w_od2[2];
    DevBuf sh_li[2], sh_ld[2], sh_pack[2], sh_gat[2], sh_gat_d[2];   // sharded k-NN: local lists, packed keys, gathered lists
    DevBuf r_qraw[2], r_q[2], r_counts[2], r_offsets[2], r_hits[2], r_slab[2], r_qlist[2], r_nlist[2], r_sums[2];  // radius pipeline workspaces
    DevBuf r_llist;               // radius_dev: the queries of a chunk whose hits the block sort orders
    // radius search of a multi-GPU handle: queries, the CSR of radius_device, the lists pulled from every shard, their merge
    DevBuf rd_q, rd_offs, rd_hits, rp_offs, rp_hits, rm_offs, rm_hits;
    // tensor path (f32 input only): per-call workspaces, see tc_filter.cuh
    DevBuf w_aaug, w_qmargin, w_trace, w_gbound;
    // pruned tensor scan (tc_prune.cuh): per-call workspaces
    DevBuf w_qs, w_seed, w_bits, w_tcnt;
    DevBuf w_bcen, w_brad, w_bmu, w_qth, w_bbits, w_bcnt, w_wslot, w_wlist, w_wbits, w_nwide;   // tile-bitmap pass: query balls, their bitmaps, wide balls

    Stream stream, s_in, s_out;   // the handle's stream; the H2D / D2H streams of the host-buffer pipelines (ensure_io)
    cudaStream_t last_stream = nullptr;

    Event ev[4];                  // timing: call (0, 1) and scan (2, 3)
    Event e_in[2], e_cmp[2], e_out[2];
    std::vector<Event> sh_ev;     // timing events of the sharded pipeline (reused)
    PinnedBuf pin_tot;            // chunk totals of the radius count pass
    PinnedBuf pin_stage[2];       // D2H staging of copy_out_staged
    Event pin_ev[2];

    explicit Engine(std::shared_ptr<DeviceTree<A>> t) : tree(std::move(t)) {}

    // A handle on `t`.  With a device, the handle's stream and timing events are created on the tree's device.
    static int open(std::shared_ptr<DeviceTree<A>> t, bool host_only, std::unique_ptr<Engine>& out) {
        std::unique_ptr<Engine> e(new Engine(std::move(t)));
        e->host_only = host_only;
        if (!host_only) {
            const int dev = e->tree->device;
            DeviceGuard g(dev);
            if (!g.ok) return fail(PN_CUDA, "no usable CUDA device (there is no CPU fallback)");
            CU(cudaDeviceGetAttribute(&e->n_sms, cudaDevAttrMultiProcessorCount, dev));
            TRY(e->stream.create());
            for (auto& x : e->ev) TRY(x.create(cudaEventDefault));
        }
        out = std::move(e);
        return PN_OK;
    }

    uint64_t device_bytes() const override {
        if (!owns_tree) return 0;
        const auto p = tree->partition();
        return tree->bytes + (p ? p->bytes : 0);
    }

    // ------------------------------------------------------------------------------------------
    template <int DVR, int K, int KIND>
    int launch_knn_t(const DeviceTree<A>& t, const KnnArgs<A>& a, dim3 grid, cudaStream_t st) {
        size_t smem = DVR < 0 ? 0 : 2 * TILE_BYTES + (DVR == 0 ? (size_t)TQ * t.ft.dpad * sizeof(A) : 0);
        auto kern = knn_tile_kernel<A, DVR, K, KIND>;
        if (smem > 32 * 1024) CU(allow_max_dynamic_smem(kern));
        kern<<<grid, TQ, smem, st>>>(a);
        CU(cudaGetLastError());
        return PN_OK;
    }
    template <int K, int KIND>
    int launch_knn_k(const DeviceTree<A>& t, const KnnArgs<A>& a, dim3 grid, cudaStream_t st) {
        switch (t.dt.dv) {
            case 1: return launch_knn_t<1, K, KIND>(t, a, grid, st);
            case 2: return launch_knn_t<2, K, KIND>(t, a, grid, st);
            case 4: return launch_knn_t<4, K, KIND>(t, a, grid, st);
            case 8: return launch_knn_t<8, K, KIND>(t, a, grid, st);
            default:
                if ((size_t)t.ft.dpad * sizeof(A) > 1024) return launch_knn_t<-1, K, KIND>(t, a, grid, st);  // wide rows: unstaged
                return launch_knn_t<0, K, KIND>(t, a, grid, st);
        }
    }
    int launch_knn(const DeviceTree<A>& t, const KnnArgs<A>& a, dim3 grid, cudaStream_t st, bool k1) {
        if (t.ft.kind == 0) return k1 ? launch_knn_k<1, 0>(t, a, grid, st) : launch_knn_k<16, 0>(t, a, grid, st);
        return k1 ? launch_knn_k<1, 1>(t, a, grid, st) : launch_knn_k<16, 1>(t, a, grid, st);
    }


    // ------------------------------------------------------------------------------------------
    // tensor path set-up (f32, d >= 8 worth of contraction): centred, augmented B operand + its TMA map
    typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                      const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                      CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
    static EncodeTiledFn encode_fn() {
        static EncodeTiledFn fn = [] {
            void* p = nullptr;
            cudaDriverEntryPointQueryResult q;
            if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess) { (void)cudaGetLastError(); p = nullptr; }
            return (EncodeTiledFn)p;
        }();
        return fn;
    }
    static int make_map(CUtensorMap* m, void* base, uint64_t rows, uint32_t box_rows, uint32_t kp) {
        EncodeTiledFn fn = encode_fn();
        if (!fn) return fail(PN_CUDA, "cuTensorMapEncodeTiled entry point not found");
        cuuint64_t dims[2] = {kp, rows};
        cuuint64_t strides[1] = {(cuuint64_t)kp * 2};
        cuuint32_t box[2] = {(cuuint32_t)tc::KC, (cuuint32_t)box_rows};
        cuuint32_t estr[2] = {1, 1};
        CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                        CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) return fail(PN_CUDA, "cuTensorMapEncodeTiled failed with code " + std::to_string((int)r));
        return PN_OK;
    }
    static constexpr size_t filter_fixed_smem(int mt, uint32_t k) {
        // alignment slack + barriers / TMEM slot + per-warp queues + per-warp top-k lists (k entries per query)
        return 1024 + 1024 + (size_t)4 * mt * 192 * 4 + (size_t)4 * mt * k * 32 * 8;
    }
    template <int DVR, int K, int MT, int NACC, int SW = tc::BN>
    int launch_filter_t(const DeviceTree<A>& t, const CUtensorMap& map_a, const tc::FilterArgs& fa, cudaStream_t st) {
        if (fa.tile_bits) return launch_filter_s<DVR, K, MT, NACC, false, SW, true>(t, map_a, fa, st);
        return fa.g_bound ? launch_filter_s<DVR, K, MT, NACC, true, SW, false>(t, map_a, fa, st) : launch_filter_s<DVR, K, MT, NACC, false, SW, false>(t, map_a, fa, st);
    }
    template <int DVR, int K, int MT, int NACC, bool SHARED, int SW, bool PRUNE>
    int launch_filter_s(const DeviceTree<A>& t, const CUtensorMap& map_a, const tc::FilterArgs& fa, cudaStream_t st) {
        const size_t smem = filter_fixed_smem(MT, fa.k) + (size_t)MT * fa.nkc * tc::A_CHUNK_BYTES + (size_t)fa.stages * fa.gs * tc::CHUNK_BYTES;
        auto kern = tc::knn_filter_kernel<DVR, K, MT, NACC, SHARED, SW, PRUNE>;
        CU(allow_max_dynamic_smem(kern));
        const unsigned gx = (fa.nq - fa.row0 + MT * tc::BM - 1) / (MT * tc::BM);
        const unsigned gy = PRUNE ? 1u : (fa.n_tiles + fa.tiles_per_split - 1) / fa.tiles_per_split;
        kern<<<dim3(gx, gy), (5 * MT + 2) * 32, smem, st>>>(map_a, t.d_baug.template as<unsigned char>(), fa);
        CU(cudaGetLastError());
        return PN_OK;
    }
    template <int K>
    int launch_filter_k(const DeviceTree<A>& t, const CUtensorMap& map_a, tc::FilterArgs& fa, cudaStream_t st) {
        const int mt = t.filter_subtiles(fa.nkc);
        const size_t budget = 224 * 1024;
        // ring groups of 16 KB (one full/empty barrier pair per group): 2 tiles at Kp = 32, 1 tile at Kp = 64, chunks beyond
        fa.gs = fa.nkc == 1 ? 2 : (fa.nkc == 2 ? 2 : 1);
        const size_t fixed = filter_fixed_smem(mt, fa.k) + (size_t)mt * fa.nkc * tc::A_CHUNK_BYTES;
        fa.stages = fixed < budget ? (uint32_t)std::min<size_t>(fa.gs > 1 ? 8 : 12, (budget - fixed) / (tc::CHUNK_BYTES * fa.gs)) : 0;
        fa.stages &= ~1u;  // even: each ring stage always belongs to the same one of the two producer warps
        if (fa.stages < 2) return fail(PN_CUDA, "tensor path: shared memory budget too small for this dimension");
        if (mt == 4) {
            // One K chunk (d <= 26): two half-tile stages per subtile (149.2 vs 151.8 ms on config 2, 21 % fewer exact
            // reranks: thresholds tightened by the first half already apply to the second).  With two or three chunks the
            // N = 64 MMAs (75 cycles against 86 for N = 128) cost more than the second stage buys: d = 64: 92.4 vs 88.4 ms.
            bool half = fa.nkc == 1;
#ifdef PN_TC_PROFILE
            if (getenv("PN_TC_HALF")) half = atoi(getenv("PN_TC_HALF")) != 0;
#endif
            if (half) {
                if (t.dt.dv == 4) return launch_filter_t<4, K, 4, 2, 64>(t, map_a, fa, st);
                if (t.dt.dv == 8) return launch_filter_t<8, K, 4, 2, 64>(t, map_a, fa, st);
                return launch_filter_t<0, K, 4, 2, 64>(t, map_a, fa, st);
            }
            if (t.dt.dv == 4) return launch_filter_t<4, K, 4, 1>(t, map_a, fa, st);
            if (t.dt.dv == 8) return launch_filter_t<8, K, 4, 1>(t, map_a, fa, st);
            return launch_filter_t<0, K, 4, 1>(t, map_a, fa, st);
        }
#if defined(PN_TC_PROFILE) || defined(PN_TC_EXPERIMENTS)
        if (mt == 3) {
            // one chunk: two half-tile stages per subtile (3 x 2 x 64 accumulator columns + 3 x 16 operand columns)
            if (fa.nkc == 1) return t.dt.dv == 4 ? launch_filter_t<4, K, 3, 2, 64>(t, map_a, fa, st) : launch_filter_t<0, K, 3, 2, 64>(t, map_a, fa, st);
            return launch_filter_t<0, K, 3, 1>(t, map_a, fa, st);
        }
#endif
        if (mt == 2) {
            if (t.dt.dv == 4) return launch_filter_t<4, K, 2, 2>(t, map_a, fa, st);
            if (t.dt.dv == 8) return launch_filter_t<8, K, 2, 2>(t, map_a, fa, st);
#if defined(PN_TC_PROFILE) || defined(PN_TC_EXPERIMENTS)
            // Experiments (diagnostic builds): the A operand in tensor memory (TS-form MMA).  scripts/mma_rate.cu, two
            // issuers, cycles per 128 accumulator columns: SS N=128 86.5 (= the 64-cycle floor + 22 of operand fetch),
            // TS N=128 70, TS N=64 78.4.  Two whole-tile stages per subtile AND the operands (2 x 2 x 128 + 2 x 72 columns at
            // d = 128) do not fit the 512 columns, and both arrangements that fit lose to the SS kernel:
            //   PN_TC_TS=2: ONE whole-tile stage per subtile: MMA and read-out of a subtile serialise, 10M x 128 scan 70.4 -> 74.0 ms
            //   PN_TC_TS=1: TWO half-tile stages per subtile (N = 64 MMAs): twice the stage hand-overs, 368 -> 436 ms
            //               (151 552 queries; profiles/r02_mma_rate.md).  Both bit-exact.
            {
                static const int ts = getenv("PN_TC_TS") ? atoi(getenv("PN_TC_TS")) : 0;
                if (ts == 1 && fa.nkc <= 8) return launch_filter_t<0, K, 2, 2, 64>(t, map_a, fa, st);
                if (ts == 2) return launch_filter_t<0, K, 2, 1>(t, map_a, fa, st);
            }
#endif
            return launch_filter_t<0, K, 2, 2>(t, map_a, fa, st);
        }
        return launch_filter_t<0, K, 1, 2>(t, map_a, fa, st);
    }

    // The members from here to knn_device_tensor serve the tensor path and are instantiated for f32 trees only (A = float,
    // V = float4): knn_device calls them from its f32 branch.

    // Prepass of the seeded scans (k <= 16): queries sorted by home bucket (self query: the stored order is that order
    // already) and every query's seed threshold from its home bucket.  *qsorted: padded query rows in sorted order; *order:
    // sorted slot -> query id (null for the self query).
    int sort_and_seed(const DeviceTree<A>& t, const A* qraw, uint32_t nq, size_t stride, uint32_t k, cudaStream_t st, bool self_query, const V** qsorted,
                      const uint32_t** order) {
        *order = nullptr;
        TRY(w_home.ensure((size_t)nq * 4));
        if (self_query) {
            TRY(w_hist.ensure((size_t)t.ft.n_buckets * 4));
            home_bucket_kernel<A><<<(nq + 127) / 128, 128, 0, st>>>(t.dt, t.d_pts.template as<V>(), nq, w_home.as<uint32_t>(), w_hist.as<uint32_t>());
            CU(cudaGetLastError());
            ++counters.kernel_launches;
            *qsorted = t.d_pts.template as<V>();
        } else {
            TRY(stage_queries(t, qraw, nq, stride, st, true));  // padded rows, home buckets, counting sort -> w_order
            TRY(w_qs.ensure((size_t)nq * t.ft.dpad * 4));
            const size_t tot = (size_t)nq * t.dt.dv;
            tc::gather_queries_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, st>>>(w_q.as<V>(), w_order.as<uint32_t>(), nq, t.dt.dv, w_qs.as<V>());
            CU(cudaGetLastError());
            ++counters.kernel_launches;
            *qsorted = w_qs.as<V>();
            *order = w_order.as<uint32_t>();
        }
        TRY(w_seed.ensure((size_t)nq * 4));
        tc::seed_bound_kernel<<<(nq + 7) / 8, 256, 0, st>>>(t.dt, *qsorted, *order, w_home.as<uint32_t>(), nq, k, w_seed.as<float>());
        CU(cudaGetLastError());
        ++counters.kernel_launches;
        return PN_OK;
    }

    // The filter arguments that come from the tree, and the query operand of the filter: the augmented FP16 rows of the
    // nq padded query rows `qpad` (w_aaug, w_qmargin) and their TMA map.  fa.part_d / part_i point at the start of
    // w_part_d / w_part_i.
    int filter_operands(const DeviceTree<A>& t, const V* qpad, uint32_t nq, cudaStream_t st, CUtensorMap* map_a, tc::FilterArgs& fa) {
        tc::build_aaug_kernel<<<(nq + 127) / 128, 128, 0, st>>>(reinterpret_cast<const float*>(qpad), t.d_center.template as<float>(), t.tscale, nq, t.ft.d,
                                                                t.ft.dpad, t.kp, t.pmax, w_aaug.as<__half>(), w_qmargin.as<float>());
        CU(cudaGetLastError());
        ++counters.kernel_launches;
        TRY(make_map(map_a, w_aaug.p, nq, tc::BM, t.kp));
        fa.t = t.dt;
        fa.q = qpad; fa.q_margin = w_qmargin.as<float>();
        fa.n_tiles = (uint32_t)((t.ft.n + tc::BN - 1) / tc::BN);
        fa.nkc = t.kp / tc::KC;
        fa.last_steps = ((t.ft.d + tc::NSLOT - 1) % tc::KC) / 16 + 1;
        fa.t2_scale = t.tscale * t.tscale * (1.0f + (float)(t.ft.d + 4) * 1.1920928955078125e-07f);
        fa.part_d = w_part_d.as<float>(); fa.part_i = w_part_i.as<uint32_t>();
        fa.counters = w_counters.as<unsigned long long>();
        return PN_OK;
    }

    // Pruned tensor k-NN (tc_prune.cuh; k <= 16): queries sorted by home bucket, seed bounds from the home bucket, one tile
    // bitmap per CTA, then ONE launch of the filter over all query groups -- the groups have lists of very different
    // lengths, so the hardware block scheduler does the load balancing that whole waves do for the dense scan.
    int knn_device_pruned(const DeviceTree<A>& t, const A* qraw, uint32_t nq, size_t stride, uint32_t k, uint32_t kstride, uint64_t* idx_out, A* dist_out, cudaStream_t st,
                          bool self_query) {
        const bool k1 = (k == 1);
        const uint32_t KP = k1 ? 1 : 16;
        const uint32_t n_tiles = (uint32_t)((t.ft.n + tc::BN - 1) / tc::BN), words = (n_tiles + 31) / 32;
        const uint32_t QT = 128u * (uint32_t)t.filter_subtiles(t.kp / tc::KC), n_qt = (nq + QT - 1) / QT;
        const V* qsorted;
        const uint32_t* order = nullptr;
        CU(cudaEventRecord(ev[2], st));   // scan_ms covers the whole scan: sort + seeds, bitmaps, filter, merge
        // PN_STAGE_TIMING=1 (diagnostic): the stages of this call timed one by one, to stderr
        static const bool stage_timing = getenv("PN_STAGE_TIMING") != nullptr;
        Event se[5];
        if (stage_timing) { for (auto& e : se) TRY(e.create(cudaEventDefault)); CU(cudaEventRecord(se[0], st)); }
        TRY(sort_and_seed(t, qraw, nq, stride, k, st, self_query, &qsorted, &order));
        if (stage_timing) CU(cudaEventRecord(se[1], st));
        TRY(w_aaug.ensure((size_t)nq * t.kp * 2));
        TRY(w_qmargin.ensure((size_t)nq * 4));
        TRY(w_bits.ensure((size_t)n_qt * words * 4));
        TRY(w_tcnt.ensure((size_t)n_qt * 4));
        TRY(w_part_d.ensure((size_t)nq * KP * 4));
        TRY(w_part_i.ensure((size_t)nq * KP * 4));
        alignas(64) CUtensorMap map_a;
        tc::FilterArgs fa{};
        TRY(filter_operands(t, qsorted, nq, st, &map_a, fa));
        {
            // tile bitmaps (tc_prune.cuh): balls of 32 sorted queries against the tile balls, wide balls refined query by query
            // PN_WIDE_DIV (diagnostic): the share of warps that may be refined query by query is 1 / PN_WIDE_DIV (0: none)
            static const int wide_div = getenv("PN_WIDE_DIV") ? atoi(getenv("PN_WIDE_DIV")) : 4;
            const uint32_t n_sub = QT / 32, n_warps = n_qt * n_sub, n_balls = 2 * n_warps;
            const uint32_t wide_cap = wide_div > 0 ? std::max<uint32_t>(1u, n_warps / (uint32_t)wide_div) : 1u;
            const size_t smem = (size_t)32 * t.dt.dv * 16;
            TRY(w_bcen.ensure((size_t)n_balls * t.ft.dpad * 4)); TRY(w_brad.ensure((size_t)n_balls * 4)); TRY(w_bmu.ensure((size_t)n_balls * 4));
            TRY(w_qth.ensure((size_t)n_warps * 32 * 4)); TRY(w_bbits.ensure((size_t)n_balls * words * 4)); TRY(w_bcnt.ensure((size_t)n_balls * 4));
            TRY(w_wslot.ensure((size_t)n_warps * 4)); TRY(w_wlist.ensure((size_t)wide_cap * 4)); TRY(w_wbits.ensure((size_t)wide_cap * words * 4));
            TRY(w_nwide.ensure(4));
            if (smem > 48u * 1024u) {
                CU(allow_max_dynamic_smem(tc::ball_tile_kernel<false>));
                CU(allow_max_dynamic_smem(tc::ball_tile_kernel<true>));
            }
            CU(cudaMemsetAsync(w_nwide.p, 0, 4, st));
            tc::warp_balls_kernel<<<(n_warps + 7) / 8, 256, 0, st>>>(qsorted, w_seed.as<float>(), nq, n_warps, t.dt.dv, w_bcen.as<float4>(), w_brad.as<float>(),
                                                                     w_bmu.as<float>(), w_qth.as<float>());
            CU(cudaGetLastError());
            tc::ball_tile_kernel<false><<<(n_balls + 31) / 32, 256, smem, st>>>(w_bcen.as<float4>(), w_brad.as<float>(), w_bmu.as<float>(), n_balls, nullptr, nullptr, 0u,
                                                                               t.d_tcen.template as<float>(), t.d_trad.template as<float>(), n_tiles, t.dt.dv, (float)t.dt.slack, words,
                                                                               w_bbits.as<uint32_t>(), w_bcnt.as<uint32_t>());
            CU(cudaGetLastError());
            tc::wide_select_kernel<<<(n_qt + 127) / 128, 128, 0, st>>>(w_bcnt.as<uint32_t>(), w_bmu.as<float>(), n_qt, n_sub, wide_div > 0 ? wide_cap : 0u, w_wslot.as<uint32_t>(),
                                                                      w_wlist.as<uint32_t>(), w_nwide.as<uint32_t>());
            CU(cudaGetLastError());
            tc::ball_tile_kernel<true><<<wide_cap, 256, smem, st>>>(qsorted, nullptr, w_qth.as<float>(), nq, w_wlist.as<uint32_t>(), w_nwide.as<uint32_t>(), wide_div > 0 ? wide_cap : 0u,
                                                                   t.d_tcen.template as<float>(), t.d_trad.template as<float>(), n_tiles, t.dt.dv, (float)t.dt.slack, words,
                                                                   w_wbits.as<uint32_t>(), nullptr);
            CU(cudaGetLastError());
            tc::group_bits_kernel<<<n_qt, 256, 0, st>>>(w_bbits.as<uint32_t>(), w_wbits.as<uint32_t>(), w_wslot.as<uint32_t>(), nq, QT, n_sub, words,
                                                        w_bits.as<uint32_t>(), w_tcnt.as<uint32_t>(), w_counters.as<unsigned long long>() + 3);
            CU(cudaGetLastError());
            counters.kernel_launches += 4;
        }
        ++counters.kernel_launches;
        if (stage_timing) CU(cudaEventRecord(se[2], st));
        fa.k = k; fa.tiles_per_split = n_tiles;
        fa.row0 = 0; fa.nq = nq; fa.g_bound = nullptr;
        fa.tile_bits = w_bits.as<uint32_t>(); fa.tile_cnt = w_tcnt.as<uint32_t>(); fa.tile_words = words; fa.seed_t2 = w_seed.as<float>();
        TRY(k1 ? launch_filter_k<1>(t, map_a, fa, st) : launch_filter_k<16>(t, map_a, fa, st));
        if (stage_timing) CU(cudaEventRecord(se[3], st));
        // results of sorted slot i belong to query order[i] (self query: to the original row of stored point i)
        CU(merge_lists<A, uint32_t>(st, w_part_d.as<A>(), w_part_i.as<uint32_t>(), 1, nq, k, idx_out, dist_out, kstride,
                                                                        0, nullptr, nullptr, self_query ? t.d_ids.template as<uint32_t>() : order));
        CU(cudaGetLastError());
        if (stage_timing) {
            CU(cudaEventRecord(se[4], st));
            CU(cudaEventSynchronize(se[4]));
            float t[4] = {0.f, 0.f, 0.f, 0.f};
            for (int i = 0; i < 4; ++i) (void)cudaEventElapsedTime(&t[i], se[i], se[i + 1]);
            fprintf(stderr, "[pn stage timing] pruned scan, %u queries, k %u: sort + seeds %.2f ms | operands + tile bitmaps %.2f ms | filter %.2f ms | merge %.2f ms\n",
                    nq, k, t[0], t[1], t[2], t[3]);
        }
        counters.kernel_launches += 2;
        counters.filter_pairs += (uint64_t)t.ft.n * nq;  // replaced by the device-side count of scanned pairs in fetch_counters
        CU(cudaEventRecord(ev[3], st));
        return PN_OK;
    }

    // tensor k-NN: same contract as knn_device
    int knn_device_tensor(const DeviceTree<A>& t, const A* qraw, uint32_t nq, size_t stride, uint32_t k, uint32_t kstride, uint64_t* idx_out, A* dist_out,
                          cudaStream_t st, bool self_query) {
        const bool k1 = (k == 1);
        const uint32_t KP = k1 ? 1 : 16;
        const uint32_t n_pass = (k + KP - 1) / KP;
        last_pruned = t.prune_on && n_pass == 1;
        last_tiles = last_pruned && t.tiles_on;
        if (last_tiles) return knn_device_pruned(t, qraw, nq, stride, k, kstride, idx_out, dist_out, st, self_query);
        // seeded scan without tile bitmaps: the dense launch plan below over the SORTED queries, every query starting
        // from its seed threshold; results return to their rows through the merge kernel's row map
        const V* qsorted = nullptr;
        const uint32_t* order = nullptr;
        CU(cudaEventRecord(ev[2], st));   // scan_ms covers the whole scan: staging, sort + seeds, filter, merge
        if (last_pruned) TRY(sort_and_seed(t, qraw, nq, stride, k, st, self_query, &qsorted, &order));
        else if (!self_query) TRY(stage_queries(t, qraw, nq, stride, st, false));
        const V* qpad = last_pruned ? qsorted : (self_query ? t.d_pts.template as<V>() : w_q.as<V>());
        TRY(w_aaug.ensure((size_t)nq * t.kp * 2));
        TRY(w_qmargin.ensure((size_t)nq * 4));
        // Launch plan.  A CTA serves QT = 128 x subtiles queries against the whole point stream, so whole waves of
        // n_sms CTAs keep every SM busy; what is left (fewer query tiles than SMs: the tail of a large batch, or
        // all of a small one) runs as a second launch whose grid.y splits the point stream S ways -- each CTA scans
        // 1/S of the points for its queries and writes its own top-k list, merged by merge_lists_kernel.
        const uint32_t n_tiles = (uint32_t)((t.ft.n + tc::BN - 1) / tc::BN);
        const uint32_t QT = 128u * (uint32_t)t.filter_subtiles(t.kp / tc::KC);
        const uint32_t n_qt = (nq + QT - 1) / QT;
        uint32_t main_qt = n_qt / (uint32_t)n_sms * (uint32_t)n_sms, tail_qt = n_qt - main_qt, S = 1, tps = n_tiles;
        if (tail_qt) {
            // S minimises the tail's duration in units of one full scan, ceil(tail_qt S / n_sms) / S, with a charge
            // of 12 % per extra split (measured: every split starts its own top-k lists, so the exact reranks of a
            // query grow ~ linearly with S, and there is one more list to merge)
            const uint32_t s_max = std::max<uint32_t>(1u, std::min<uint32_t>({std::max<uint32_t>(16u, (uint32_t)n_sms / tail_qt), n_tiles / 64u, (uint32_t)MAX_LISTS}));
            double best = 1e30;
            for (uint32_t c = 1; c <= s_max; ++c) {
                const double cost = (double)((tail_qt * c + n_sms - 1) / n_sms) / c * (1.0 + 0.12 * (c - 1));
                if (cost < best) { best = cost; S = c; }
            }
            tps = (n_tiles + S - 1) / S;
            S = (n_tiles + tps - 1) / tps;  // every split non-empty
        }
        if (S == 1) { main_qt = n_qt; tail_qt = 0; }
        const uint32_t q_main = (uint32_t)std::min<uint64_t>((uint64_t)main_qt * QT, nq), q_tail = nq - q_main;
        TRY(w_part_d.ensure(((size_t)q_main + (size_t)S * q_tail) * KP * 4));
        TRY(w_part_i.ensure(((size_t)q_main + (size_t)S * q_tail) * KP * 4));
        if (n_pass > 1) { TRY(w_floor_d.ensure((size_t)nq * 4)); TRY(w_floor_i.ensure((size_t)nq * 4)); }
        alignas(64) CUtensorMap map_a;
        tc::FilterArgs fa0{};
        TRY(filter_operands(t, qpad, nq, st, &map_a, fa0));
        for (uint32_t p = 0; p < n_pass; ++p) {
            const uint32_t kk = std::min(KP, k - p * KP);
            tc::FilterArgs fa = fa0;
            fa.k = kk;
            fa.floor_d = p ? w_floor_d.as<float>() : nullptr; fa.floor_i = p ? w_floor_i.as<uint32_t>() : nullptr;
#ifdef PN_TC_PROFILE
            fa.dbg = getenv("PN_TC_DEBUG") ? (uint32_t)atoi(getenv("PN_TC_DEBUG")) : 0u;
            if (getenv("PN_TC_TRACE")) {
                TRY(w_trace.ensure(12 * 64 * 4 * 8));
                CU(cudaMemsetAsync(w_trace.p, 0, 12 * 64 * 4 * 8, st));
                fa.trace = w_trace.as<long long>();
                fa.trace_t0 = getenv("PN_TC_TRACE_T0") ? (uint32_t)atoi(getenv("PN_TC_TRACE_T0")) : 2000u;
            }
#endif
            A* fl_d = n_pass > 1 ? w_floor_d.as<A>() : nullptr;
            uint32_t* fl_i = n_pass > 1 ? w_floor_i.as<uint32_t>() : nullptr;
            const uint32_t* rmap = self_query ? t.d_ids.template as<uint32_t>() : order;
            fa.seed_t2 = last_pruned ? w_seed.as<float>() : nullptr;
            if (q_main) {
                fa.row0 = 0; fa.nq = q_main; fa.tiles_per_split = n_tiles; fa.g_bound = nullptr;
                TRY(k1 ? launch_filter_k<1>(t, map_a, fa, st) : launch_filter_k<16>(t, map_a, fa, st));
                CU(merge_lists<A, uint32_t>(st, w_part_d.as<A>(), w_part_i.as<uint32_t>(), 1, q_main, kk, idx_out, dist_out, kstride, p * KP, fl_d, fl_i, rmap));
                CU(cudaGetLastError());
                counters.kernel_launches += 2;
            }
            if (q_tail) {
                fa.row0 = q_main; fa.nq = nq; fa.tiles_per_split = tps;
                if (S > 1) {  // the splits of a query share their k-th bounds (initialised to a huge finite float)
                    TRY(w_gbound.ensure((size_t)q_tail * 4));
                    CU(cudaMemsetAsync(w_gbound.p, 0x7f, (size_t)q_tail * 4, st));
                    fa.g_bound = w_gbound.as<float>();
                }
                fa.part_d = w_part_d.as<float>() + (size_t)q_main * kk; fa.part_i = w_part_i.as<uint32_t>() + (size_t)q_main * kk;
                TRY(k1 ? launch_filter_k<1>(t, map_a, fa, st) : launch_filter_k<16>(t, map_a, fa, st));
                // with a row map (self query) the merge addresses output rows absolutely; otherwise the outputs are offset
                CU(merge_lists<A, uint32_t>(st, reinterpret_cast<const A*>(fa.part_d), fa.part_i, S, q_tail, kk, rmap ? idx_out : idx_out + (size_t)q_main * kstride,
                    rmap ? dist_out : dist_out + (size_t)q_main * kstride, kstride, p * KP, fl_d ? fl_d + q_main : nullptr,
                    fl_i ? fl_i + q_main : nullptr, rmap ? rmap + q_main : nullptr));
                CU(cudaGetLastError());
                counters.kernel_launches += 2;
            }
            counters.filter_pairs += (uint64_t)t.ft.n * nq;
        }
        CU(cudaEventRecord(ev[3], st));
        return PN_OK;
    }

    int use_stream(cudaStream_t st) {
        if (last_stream && last_stream != st) CU(cudaStreamSynchronize(last_stream));
        last_stream = st;
        return PN_OK;
    }

    // queries (raw rows on the device) -> zero-padded rows + tile order
    int stage_queries(const DeviceTree<A>& t, const A* qraw, uint32_t nq, size_t stride, cudaStream_t st, bool sort) {
        TRY(w_q.ensure((size_t)nq * t.ft.dpad * sizeof(A)));
        const size_t tot = (size_t)nq * t.ft.dpad;
        pad_queries_kernel<A><<<(unsigned)((tot + 255) / 256), 256, 0, st>>>(qraw, stride, nq, t.ft.d, t.ft.dpad, w_q.as<A>());
        CU(cudaGetLastError());
        ++counters.kernel_launches;
        if (!sort) return PN_OK;
        TRY(w_home.ensure((size_t)nq * 4));
        TRY(w_order.ensure((size_t)nq * 4));
        TRY(w_hist.ensure((size_t)t.ft.n_buckets * 4));
        TRY(w_cursor.ensure((size_t)t.ft.n_buckets * 4));
        CU(cudaMemsetAsync(w_hist.p, 0, (size_t)t.ft.n_buckets * 4, st));
        home_bucket_kernel<A><<<(nq + 127) / 128, 128, 0, st>>>(t.dt, w_q.as<V>(), nq, w_home.as<uint32_t>(), w_hist.as<uint32_t>());
        CU(cudaGetLastError());
        exclusive_scan_kernel<<<1, 1024, 0, st>>>(w_hist.as<uint32_t>(), w_cursor.as<uint32_t>(), t.ft.n_buckets);
        CU(cudaGetLastError());
        scatter_order_kernel<<<(nq + 255) / 256, 256, 0, st>>>(w_home.as<uint32_t>(), w_cursor.as<uint32_t>(), nq, w_order.as<uint32_t>());
        CU(cudaGetLastError());
        counters.kernel_launches += 3;
        return PN_OK;
    }

    // k-NN for nq queries whose raw rows are already on the device; results to device buffers
    // self_query: the queries are the stored points themselves, already padded, resident and in bucket
    // order (perfect tile coherence); results are written to the ORIGINAL row of each point
    int knn_device(const DeviceTree<A>& t, const A* qraw, uint32_t nq, size_t stride, uint32_t k_req, uint64_t* idx_out, A* dist_out, cudaStream_t st,
                   bool self_query = false) {
        if (!self_query) {   // batches of queries are answered from the partition when the tensor path scans it (DeviceTree::part)
            const auto p = t.partition();
            if (p && p->tensor_ready) return knn_device(*p, qraw, nq, stride, k_req, idx_out, dist_out, st);
        }
        // k > n: only n neighbours exist; scan for those and pad the remaining columns directly
        const uint32_t kstride = k_req, k = (uint32_t)std::min<uint64_t>(k_req, t.ft.n);
        if (k < kstride) {
            const size_t tot = (size_t)nq * (kstride - k);
            pad_rows_kernel<A><<<(unsigned)((tot + 255) / 256), 256, 0, st>>>(idx_out, dist_out, nq, kstride, k);
            CU(cudaGetLastError());
            ++counters.kernel_launches;
        }
        // AUTO: with the point stream split over the SMs the tensor path wins at every batch size measured (uniform 1M x 16:
        // 1 query 0.43 vs 0.80 ms, 1024 queries 1.2 vs 8.3 ms; 1M x 128: 0.43 vs 3.8 ms and 1.3 vs 31.8 ms,
        // scripts/small_batch.py), so AUTO uses it for every batch size whenever the tree is tensor-eligible (f32, d >= 16).
        // The pruned scan can still win for single queries on tightly clustered data (it touches a few buckets only):
        // PN_ALGO_SIMT selects it.
        last_used_tensor = t.tensor_ready;   // only ever set on f32 trees (DeviceTree::prepare_tensor)
        if constexpr (sizeof(A) == 4) {
            if (last_used_tensor) return knn_device_tensor(t, qraw, nq, stride, k, kstride, idx_out, dist_out, st, self_query);
        }
        // narrow rows of a ball tree: one warp per query (knn_warp_kernel) -- every query walks its own few buckets
        if (t.ft.kind == 0 && t.ft.d <= 8 && t.dt.dv <= 4) {
            const bool wsort = !self_query && t.ft.n_buckets > 1 && nq >= 16384;   // neighbouring warps then share buckets in L1 / L2
            if (!self_query) TRY(stage_queries(t, qraw, nq, stride, st, wsort));
            const uint32_t WP = 32, w_pass = (k + WP - 1) / WP;
            if (w_pass > 1) { TRY(w_floor_d.ensure((size_t)nq * sizeof(A))); TRY(w_floor_i.ensure((size_t)nq * 4)); }
            CU(cudaEventRecord(ev[2], st));
            for (uint32_t p = 0; p < w_pass; ++p) {
                WarpKnnArgs<A> a{};
                a.t = t.dt; a.q = self_query ? t.d_pts.template as<V>() : w_q.as<V>();
                a.qorder = wsort ? w_order.as<uint32_t>() : nullptr;
                a.row_map = self_query ? t.d_ids.template as<uint32_t>() : nullptr;
                a.nq = nq; a.k = std::min(WP, k - p * WP);
                a.out_i = idx_out; a.out_d = dist_out; a.out_stride = kstride; a.out_off = p * WP;
                a.floor_d = w_pass > 1 ? w_floor_d.as<A>() : nullptr; a.floor_i = w_pass > 1 ? w_floor_i.as<uint32_t>() : nullptr;
                a.pass = p;
                a.counters = w_counters.as<unsigned long long>();
                knn_warp_kernel<A><<<(nq + 7) / 8, 256, 0, st>>>(a);
                CU(cudaGetLastError());
                ++counters.kernel_launches;
            }
            CU(cudaEventRecord(ev[3], st));
            return PN_OK;
        }
        const bool sort = !self_query && t.ft.n_buckets > 1 && nq > (uint32_t)TQ;
        if (!self_query) TRY(stage_queries(t, qraw, nq, stride, st, sort));
        const uint32_t tiles = (nq + TQ - 1) / TQ;
        uint32_t sl = 0;
        while (((uint64_t)tiles << sl) < 2ull * n_sms && sl < t.ft.L && (2u << sl) <= (uint32_t)MAX_LISTS) ++sl;
        const uint32_t n_splits = 1u << sl;
        const bool k1 = (k == 1);
        const uint32_t KP = k1 ? 1 : 16;
        const uint32_t n_pass = (k + KP - 1) / KP;
        TRY(w_part_d.ensure((size_t)n_splits * nq * KP * sizeof(A)));
        TRY(w_part_i.ensure((size_t)n_splits * nq * KP * 4));
        if (n_pass > 1) { TRY(w_floor_d.ensure((size_t)nq * sizeof(A))); TRY(w_floor_i.ensure((size_t)nq * 4)); }
        CU(cudaEventRecord(ev[2], st));
        for (uint32_t p = 0; p < n_pass; ++p) {
            const uint32_t kk = std::min(KP, k - p * KP);
            KnnArgs<A> a{};
            a.t = t.dt; a.q = self_query ? t.d_pts.template as<V>() : w_q.as<V>(); a.qorder = sort ? w_order.as<uint32_t>() : nullptr;
            a.nq = nq; a.k = kk; a.split_level = sl;
            a.part_d = w_part_d.as<A>(); a.part_i = w_part_i.as<uint32_t>();
            a.floor_d = p ? w_floor_d.as<A>() : nullptr; a.floor_i = p ? w_floor_i.as<uint32_t>() : nullptr;
            a.counters = w_counters.as<unsigned long long>();
            if (n_splits > 1) {   // the splits of a query share their k-th bounds (initialised to a huge finite value)
                TRY(w_gbound.ensure((size_t)nq * sizeof(A)));
                CU(cudaMemsetAsync(w_gbound.p, 0x7f, (size_t)nq * sizeof(A), st));
                a.g_bound = w_gbound.as<A>();
            }
            TRY(launch_knn(t, a, dim3(tiles, n_splits), st, k1));
            CU(merge_lists<A, uint32_t>(st, w_part_d.as<A>(), w_part_i.as<uint32_t>(), n_splits, nq, kk, idx_out, dist_out, kstride, p * KP,
                n_pass > 1 ? w_floor_d.as<A>() : nullptr, n_pass > 1 ? w_floor_i.as<uint32_t>() : nullptr,
                self_query ? t.d_ids.template as<uint32_t>() : nullptr));
            CU(cudaGetLastError());
            counters.kernel_launches += 2;
        }
        CU(cudaEventRecord(ev[3], st));
        return PN_OK;
    }

    // One query call on this handle, made after the call's argument checks: holds the handle's mutex and makes the tree's
    // device current until the call returns.  open() selects the call's stream (after the handle's previous stream, see
    // use_stream) and starts a new set of counters; start() zeroes the device-side counters and starts device_ms;
    // finish() ends device_ms and fetches the device-side counters, or for an unsynchronised call only sets `queries`.
    struct Call {
        Engine& e;
        std::lock_guard<std::mutex> lk;
        DeviceGuard g;
        cudaStream_t st = nullptr;
        explicit Call(Engine& en) : e(en), lk(en.mu), g(en.tree->device) {}
        int device() const { return g.ok ? PN_OK : fail(PN_CUDA, "cudaSetDevice failed"); }
        int open(cudaStream_t s) {
            TRY(device());
            st = s;
            TRY(e.use_stream(st));
            e.counters = pn_counters{};
            return PN_OK;
        }
        int start() {
            TRY(e.w_counters.ensure(256));
            CU(cudaMemsetAsync(e.w_counters.p, 0, 256, st));
            CU(cudaEventRecord(e.ev[0], st));
            return PN_OK;
        }
        int finish(uint64_t nq, bool sync = true) {
            CU(cudaEventRecord(e.ev[1], st));
            if (sync) return e.fetch_counters(st, nq);
            e.counters.queries = nq;
            return PN_OK;
        }
    };

    int fetch_counters(cudaStream_t st, uint64_t nq) {
        unsigned long long c[4] = {0, 0, 0, 0};
        CU(cudaMemcpyAsync(c, w_counters.p, 32, cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
#ifdef PN_TC_PROFILE
        if (last_used_tensor && w_counters.cap >= 256) {
            unsigned long long pc[20];
            CU(cudaMemcpy(pc, (char*)w_counters.p + 64, sizeof(pc), cudaMemcpyDeviceToHost));
            const auto p = tree->partition();
            const DeviceTree<A>& t = p && p->tensor_ready ? *p : *tree;
            const double tiles = (double)((t.ft.n + tc::BN - 1) / tc::BN) * (double)((nq + 128 * t.filter_subtiles(t.kp / tc::KC) - 1) / (128 * t.filter_subtiles(t.kp / tc::KC)));
            if (getenv("PN_TC_TRACE") && w_trace.p) {
                std::vector<long long> tr(12 * 64 * 4);
                CU(cudaMemcpy(tr.data(), w_trace.p, tr.size() * 8, cudaMemcpyDeviceToHost));
                if (FILE* f = fopen(getenv("PN_TC_TRACE"), "wb")) { fwrite(tr.data(), 8, tr.size(), f); fclose(f); }
            }
            fprintf(stderr, "[tc profile] cycles/tile  MMA thread: wait tempty %.0f | wait full %.0f | issue+commit %.0f   epilogue warp: wait tfull %.0f | TMEM read-out %.0f | scan+push %.0f | drain+margin %.0f   producer 0: wait empty %.0f | issue %.0f\n",
                    pc[0] / tiles, pc[1] / tiles, pc[2] / tiles, pc[6] / tiles, pc[7] / tiles, pc[8] / tiles, pc[9] / tiles, pc[12] / tiles, pc[13] / tiles);
        }
#endif
        counters.queries = nq;
        counters.pairs = last_used_tensor ? counters.filter_pairs : c[0];
        if (last_used_tensor && last_tiles) {  // the pruned scan counts the (query, point) pairs of the tiles it really visits
            counters.pairs = std::min<uint64_t>(c[3], counters.filter_pairs);
            counters.filter_pairs = counters.pairs;
        }
        counters.node_visits = c[1];
        counters.rerank_pairs = c[2];
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, ev[0], ev[1]) == cudaSuccess) counters.device_ms = ms; else (void)cudaGetLastError();
        if (cudaEventElapsedTime(&ms, ev[2], ev[3]) == cudaSuccess) counters.scan_ms = ms; else (void)cudaGetLastError();
        return PN_OK;
    }

    int check_query_args(const void* q, size_t nq, size_t stride) {
        if (host_only) return fail(PN_CUDA, "tree was built with PN_FLAG_HOST_ONLY: no device, and there is no CPU fallback");
        if (nq && !q) return fail(PN_BAD_ARG, "queries is null");
        if (nq >= (1ull << 32)) return fail(PN_BAD_ARG, "nq must be < 2^32 per call");
        if (nq > 1 && stride < tree->ft.d) return fail(PN_BAD_ARG, "q_row_stride < dimension");
        return PN_OK;
    }
    // k is a u32 inside the engine; the result buffers of a chunk (w_out_*) are k * 12..16 bytes per query
    static int check_k(size_t k) {
        if (k > (1u << 20)) return fail(PN_BAD_ARG, "k must be <= 2^20");
        return PN_OK;
    }

    // The pipeline streams and events, all or nothing: e_out[1] is created last, so while it is null a later call
    // creates the whole set again.
    int ensure_io() {
        if (e_out[1]) return PN_OK;
        TRY(s_in.create());
        TRY(s_out.create());
        for (int i = 0; i < 2; ++i)
            for (Event* e : {&e_in[i], &e_cmp[i], &e_out[i]}) TRY(e->create(cudaEventDisableTiming));
        return PN_OK;
    }
    // Chunk boundaries of a host-buffer call: whole waves of the scan (n_sms CTAs x the scan's queries per CTA).  Two
    // chunks are enough to hide the copies (H2D of the second and D2H of the first run under the other's kernels) and keep
    // the per-chunk costs (query staging, sort, seeds, the drain of a launch's last wave, a partial last wave) small;
    // chunks are capped at 2^20 queries (workspace size).  Measured alternative: one-wave first and last chunks (less
    // exposed copy) -- the same 107.9 ms on config 2 and 2770 instead of 2724 ms on 10M x 128 (scripts/e2e_chunks.py).
    std::vector<size_t> host_chunks(size_t nq) const {
        const size_t wave = (size_t)n_sms * tree->query_tile();
        std::vector<size_t> b{0};
        if (nq >= 4 * wave) {
            const size_t half = std::min<size_t>(((nq + 1) / 2 + wave - 1) / wave * wave, ((size_t)1 << 20) / wave * wave);
            for (size_t x = half; x < nq; x += half) b.push_back(x);
        }
        b.push_back(nq);
        return b;
    }

    int knn_host(const void* qv, size_t nq, size_t stride, size_t k, uint64_t* idx, void* distv) override {
        TRY(check_query_args(qv, nq, stride));
        TRY(check_k(k));
        if (k == 0 || nq == 0) return PN_OK;  // src/ball_tree.rs:106-108
        if (!idx || !distv) return fail(PN_BAD_ARG, "output buffer is null");
        Call call(*this);
        const cudaStream_t st = stream;
        TRY(call.open(st));
        const A* q = (const A*)qv;
        A* dist = (A*)distv;
        TRY(ensure_io());
        const std::vector<size_t> cb = host_chunks(nq);
        const size_t n_chunks = cb.size() - 1;
        size_t chunk = 0;   // the largest chunk sizes the buffers
        for (size_t c = 0; c < n_chunks; ++c) chunk = std::max(chunk, cb[c + 1] - cb[c]);
        const size_t spitch = std::max<size_t>(stride, tree->ft.d) * sizeof(A);  // a single row may come with any stride
        // every allocation happens before the first copy is enqueued (cudaMalloc synchronises the device)
        for (int b = 0; b < (n_chunks > 1 ? 2 : 1); ++b) {
            TRY(w_qraw2[b].ensure(chunk * tree->ft.d * sizeof(A)));
            TRY(w_oi2[b].ensure(chunk * k * 8));
            TRY(w_od2[b].ensure(chunk * k * sizeof(A)));
        }
        TRY(call.start());
        CU(cudaStreamWaitEvent(s_in, ev[0], 0));
        // Enqueue order: H2D(c), kernels(c), then D2H(c-1).  With pageable host memory a D2H copy blocks the host until it
        // is done, so it is issued only after the next chunk's kernels are already queued behind it on the device.
        auto d2h = [&](size_t c) -> int {
            const int b = (int)(c & 1);
            const size_t q0 = cb[c];
            const uint32_t cq = (uint32_t)(cb[c + 1] - q0);
            CU(cudaStreamWaitEvent(s_out, e_cmp[b], 0));
            TRY(results_to_host(idx + q0 * k, dist + q0 * k, w_oi2[b].as<uint64_t>(), w_od2[b].as<A>(), (size_t)cq * k, s_out));
            CU(cudaEventRecord(e_out[b], s_out));
            counters.d2h_bytes += (uint64_t)cq * k * (8 + sizeof(A));
            return PN_OK;
        };
        for (size_t c = 0; c < n_chunks; ++c) {
            const int b = (int)(c & 1);
            const size_t q0 = cb[c];
            const uint32_t cq = (uint32_t)(cb[c + 1] - q0);
            // H2D: the raw-query buffer is free once the kernels of chunk c-2 are done
            if (c >= 2) CU(cudaStreamWaitEvent(s_in, e_cmp[b], 0));
            CU(cudaMemcpy2DAsync(w_qraw2[b].p, tree->ft.d * sizeof(A), q + q0 * stride, spitch, tree->ft.d * sizeof(A), cq, cudaMemcpyHostToDevice, s_in));
            CU(cudaEventRecord(e_in[b], s_in));
            // kernels: need the queries, and the result buffers back from the D2H of chunk c-2
            CU(cudaStreamWaitEvent(st, e_in[b], 0));
            if (c >= 2) CU(cudaStreamWaitEvent(st, e_out[b], 0));
            TRY(knn_device(*tree, w_qraw2[b].as<A>(), cq, tree->ft.d, (uint32_t)k, w_oi2[b].as<uint64_t>(), w_od2[b].as<A>(), st));
            CU(cudaEventRecord(e_cmp[b], st));
            counters.h2d_bytes += (uint64_t)cq * tree->ft.d * sizeof(A);
            if (c >= 1) TRY(d2h(c - 1));
        }
        TRY(d2h(n_chunks - 1));
        // the call ends when the last results are on the host: the tree's stream joins the D2H stream
        CU(cudaStreamWaitEvent(st, e_out[(n_chunks - 1) & 1], 0));
        if (n_chunks > 1) CU(cudaStreamWaitEvent(st, e_out[(n_chunks - 2) & 1], 0));
        return call.finish(nq);
    }

    int knn_dev(const void* qv, size_t nq, size_t stride, size_t k, uint64_t* idx, void* distv, cudaStream_t st, bool sync) override {
        TRY(check_query_args(qv, nq, stride));
        TRY(check_k(k));
        if (k == 0 || nq == 0) return PN_OK;
        if (!idx || !distv) return fail(PN_BAD_ARG, "output buffer is null");
        Call call(*this);
        TRY(call.open(st ? st : (cudaStream_t)stream));
        TRY(call.start());
        TRY(knn_device(*tree, (const A*)qv, (uint32_t)nq, stride, (uint32_t)k, idx, (A*)distv, call.st));
        return call.finish(nq, sync);
    }

    // Device -> host through two pinned buffers, in pieces of PIN_BYTES: while piece p+1 is in flight, piece p is handed
    // to land(off, piece, lo, hi), which moves bytes [lo, hi) of the piece that starts at byte `off` of the copy to their
    // destination.  Up to `max_threads` host threads share a piece, in slices that are multiples of `align` bytes.  Into
    // freshly allocated memory, page faults and the host-side step, not the DMA, are the slow part.
    template <typename Land>
    int copy_out_staged(const void* src_dev, size_t bytes, cudaStream_t st, unsigned max_threads, size_t align, Land land) {
        if (bytes == 0) return PN_OK;
        for (int i = 0; i < 2; ++i) {
            if (!pin_stage[i]) TRY(pin_stage[i].create(PIN_BYTES));
            if (!pin_ev[i]) TRY(pin_ev[i].create(cudaEventDisableTiming));
        }
        const size_t pieces = (bytes + PIN_BYTES - 1) / PIN_BYTES;
        auto issue = [&](size_t p) -> int {
            const size_t off = p * PIN_BYTES, cnt = std::min(PIN_BYTES, bytes - off);
            CU(cudaMemcpyAsync(pin_stage[p & 1], (const unsigned char*)src_dev + off, cnt, cudaMemcpyDeviceToHost, st));
            CU(cudaEventRecord(pin_ev[p & 1], st));
            return PN_OK;
        };
        TRY(issue(0));
        const unsigned nt = std::max(1u, std::min(max_threads, std::thread::hardware_concurrency() / 2));
        for (size_t p = 0; p < pieces; ++p) {
            CU(cudaEventSynchronize(pin_ev[p & 1]));
            if (p + 1 < pieces) TRY(issue(p + 1));  // the other buffer was consumed in the previous iteration
            const size_t off = p * PIN_BYTES, cnt = std::min(PIN_BYTES, bytes - off);
            const unsigned char* sp = pin_stage[p & 1].template as<unsigned char>();
            const size_t chunk = ((cnt + nt - 1) / nt + align - 1) / align * align;
            std::vector<std::thread> th;
            for (unsigned t = 1; t < nt; ++t) {
                const size_t b = t * chunk, e = std::min(cnt, b + chunk);
                if (b < e) th.emplace_back([=] { land(off, sp, b, e); });
            }
            land(off, sp, 0, std::min(cnt, chunk));
            for (auto& x : th) x.join();
        }
        return PN_OK;
    }
    static bool is_pageable(const void* p) {
        cudaPointerAttributes at{};
        if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { (void)cudaGetLastError(); return true; }
        return at.type == cudaMemoryTypeUnregistered;
    }
    // The k-NN results of one call (count = queries x k) from the device to the caller's host buffers.  Pageable
    // destinations of 4 MiB of indices and more go through the pinned staging, copied in page-aligned slices on up to 8
    // host threads: the driver's own staged copy runs at about 4 GB/s into freshly allocated pages (it faults them in one
    // by one).
    int results_to_host(uint64_t* idx, A* dist, const uint64_t* idx_dev, const A* dist_dev, size_t count, cudaStream_t st) {
        if (count * 8 >= ((size_t)4 << 20) && (is_pageable(idx) || is_pageable(dist))) {
            auto bytes_to = [](void* dst) {
                return [dst](size_t off, const unsigned char* sp, size_t lo, size_t hi) { memcpy((unsigned char*)dst + off + lo, sp + lo, hi - lo); };
            };
            TRY(copy_out_staged(idx_dev, count * 8, st, 8, 4096, bytes_to(idx)));
            TRY(copy_out_staged(dist_dev, count * sizeof(A), st, 8, 4096, bytes_to(dist)));
        } else {
            CU(cudaMemcpyAsync(idx, idx_dev, count * 8, cudaMemcpyDeviceToHost, st));
            CU(cudaMemcpyAsync(dist, dist_dev, count * sizeof(A), cudaMemcpyDeviceToHost, st));
        }
        return PN_OK;
    }

    // every stored point is a query (benches/ball_tree.rs:53-59): no H2D at all
    int knn_self(size_t k, uint64_t* idx, void* distv, bool dev, cudaStream_t st, bool sync) override {
        if (host_only) return fail(PN_CUDA, "tree was built with PN_FLAG_HOST_ONLY: no device, and there is no CPU fallback");
        if (tree->ft.n != tree->ft.n_total) return fail(PN_BAD_ARG, "self-query needs the whole point set in this handle (not a shard)");
        TRY(check_k(k));
        if (k == 0) return PN_OK;
        if (!idx || !distv) return fail(PN_BAD_ARG, "output buffer is null");
        Call call(*this);
        if (!st || !dev) st = stream;
        TRY(call.open(st));
        const uint32_t nq = (uint32_t)tree->ft.n;
        uint64_t* oi = idx; A* od = (A*)distv;
        if (!dev) {
            TRY(w_out_i.ensure((size_t)nq * k * 8));
            TRY(w_out_d.ensure((size_t)nq * k * sizeof(A)));
            oi = w_out_i.as<uint64_t>(); od = w_out_d.as<A>();
        }
        TRY(call.start());
        TRY(knn_device(*tree, tree->d_pts.template as<A>(), nq, tree->ft.dpad, (uint32_t)k, oi, od, st, true));
        if (!dev) {
            TRY(results_to_host(idx, (A*)distv, oi, od, (size_t)nq * k, st));
            counters.d2h_bytes = (uint64_t)nq * k * (8 + sizeof(A));
        }
        return call.finish(nq, sync || !dev);
    }

    // Result buffers of the radius call are handed to the caller (released with pn_free = free()).  Large ones are
    // 2 MiB-aligned and advised as huge pages: writing hundreds of MB of freshly mapped memory is otherwise dominated by
    // 4 KiB page faults.
    static void* result_alloc(size_t bytes) {
        if (bytes < (8u << 20)) return malloc(bytes ? bytes : 8);
        const size_t al = 2u << 20;
        void* p = aligned_alloc(al, (bytes + al - 1) / al * al);
#ifdef MADV_HUGEPAGE
        if (p) madvise(p, (bytes + al - 1) / al * al, MADV_HUGEPAGE);
#endif
        return p;
    }

    // the host step of copy_out_staged for radius hits: u32 on the device, u64 at dst
    static auto widen_to(uint64_t* dst) {
        return [dst](size_t off, const unsigned char* sp, size_t lo, size_t hi) {
            const uint32_t* s32 = (const uint32_t*)sp;
            uint64_t* d64 = dst + off / 4;
            for (size_t i = lo / 4; i < hi / 4; ++i) d64[i] = s32[i];
        };
    }

    // ---- the device stages of radius search over one chunk of at most `chunk` queries, in workspace set b, on stream s.
    // Split in two because the host must size the hit buffer from the count pass before the fill pass runs.
    static constexpr uint32_t RADIUS_WPB = 8;   // warps (queries) per block of the traversal, compaction and sort
    int radius_workspace(const DeviceTree<A>& t, int n_sets, size_t chunk) {
        for (int b = 0; b < n_sets; ++b) {
            TRY(r_q[b].ensure(chunk * t.ft.dpad * sizeof(A)));
            TRY(r_counts[b].ensure(chunk * 4));
            TRY(r_offsets[b].ensure((chunk + 1) * 8));
            TRY(r_sums[b].ensure((chunk / SCAN_BLOCK + 1) * 8));
            TRY(r_slab[b].ensure(chunk * RADIUS_CAP * 4));
            TRY(r_qlist[b].ensure(chunk * 4));
            TRY(r_nlist[b].ensure(16));
        }
        return PN_OK;
    }
    // pad the queries (row stride q_stride elements), count traversal with the first RADIUS_CAP hits of each query in its
    // slab, chunk-local offsets (r_offsets[b][cq] is the chunk's total).  radius_dev passes `offs`, the caller's array at
    // the chunk's first query, and from the second chunk on `base` == offs: the offsets are then absolute.
    int radius_count(const DeviceTree<A>& t, int b, const A* q, size_t q_stride, uint32_t cq, A r, cudaStream_t s,
                     uint64_t* offs = nullptr, const uint64_t* base = nullptr) {
        const size_t tot = (size_t)cq * t.ft.dpad;
        pad_queries_kernel<A><<<(unsigned)((tot + 255) / 256), 256, 0, s>>>(q, q_stride, cq, t.ft.d, t.ft.dpad, r_q[b].as<A>());
        CU(cudaGetLastError());
        const unsigned blocks = (cq + RADIUS_WPB - 1) / RADIUS_WPB;
        CU(cudaMemsetAsync(r_nlist[b].p, 0, 8, s));   // the lengths of the two lists of radius_fill
        radius_kernel<A, 0><<<blocks, RADIUS_WPB * 32, 0, s>>>(t.dt, r_q[b].as<V>(), cq, r, r_counts[b].as<uint32_t>(), nullptr, r_slab[b].as<uint32_t>(),
                                                              w_counters.as<unsigned long long>());
        CU(cudaGetLastError());
        const unsigned sblocks = std::max(1u, (cq + SCAN_BLOCK - 1) / SCAN_BLOCK);
        scan_sums_kernel<<<sblocks, 1024, 0, s>>>(r_counts[b].as<uint32_t>(), cq, r_sums[b].as<unsigned long long>());
        offsets_scan_kernel<<<sblocks, 1024, 0, s>>>(r_counts[b].as<uint32_t>(), r_sums[b].as<unsigned long long>(),
                                                     offs ? offs : r_offsets[b].as<uint64_t>(), cq, base);
        CU(cudaGetLastError());
        counters.kernel_launches += 4;
        return PN_OK;
    }
    // slabs -> hits at the offsets, second traversal of the queries that overflowed their slab, per-query ascending sort.
    // Host pipelines: chunk-local offsets (r_offsets[b]), hits[0 .. ctotal) u32, and the block sort is launched when the
    // chunk's total says some list may need it.  radius_dev: `offs` as in radius_count, hits the caller's u64 array, only
    // the queries whose segment ends at or below `capacity` are written, and the block sort always runs, over the list of
    // long segments the compaction builds (ctotal is not known on the host).
    template <typename I>
    int radius_fill(const DeviceTree<A>& t, int b, uint32_t cq, A r, uint64_t ctotal, I* hits, cudaStream_t s,
                    const uint64_t* offs = nullptr, uint64_t capacity = ~0ull) {
        const unsigned blocks = (cq + RADIUS_WPB - 1) / RADIUS_WPB;
        const uint64_t* o = offs ? offs : r_offsets[b].as<uint64_t>();
        uint32_t* n_lists = r_nlist[b].as<uint32_t>();   // [0]: slab overflows, [1]: long segments (radius_dev)
        uint32_t* llist = offs ? r_llist.as<uint32_t>() : nullptr;
        compact_hits_kernel<I><<<blocks, RADIUS_WPB * 32, 0, s>>>(r_slab[b].as<uint32_t>(), r_counts[b].as<uint32_t>(), o, cq, hits,
                                                                  r_qlist[b].as<uint32_t>(), n_lists, capacity, llist, n_lists + 1);
        CU(cudaGetLastError());
        // second traversal for the queries that overflowed their slab only (warps past the list length exit at once)
        radius_kernel<A, 1, I><<<blocks, RADIUS_WPB * 32, 0, s>>>(t.dt, r_q[b].as<V>(), cq, r, nullptr, o, hits,
                                                                 nullptr, r_qlist[b].as<uint32_t>(), n_lists);
        CU(cudaGetLastError());
        segment_sort_kernel<I><<<blocks, RADIUS_WPB * 32, 0, s>>>(o, hits, cq, capacity);
        CU(cudaGetLastError());
        if (llist || ctotal > SORT_WARP_MAX) {  // some hit list may be longer than a warp should sort: one block per such query
            segment_sort_large_kernel<I><<<std::min<uint32_t>(cq, 8u * (uint32_t)n_sms), 256, 0, s>>>(o, hits, cq, llist, n_lists + 1);
            CU(cudaGetLastError());
            ++counters.kernel_launches;
        }
        counters.kernel_launches += 3;
        return PN_OK;
    }

    // Radius search of nq queries already on the tree's device (row stride `stride` elements), called under an open Call
    // on its stream st: the CSR result is left in rd_offs (u64, nq + 1 entries over the whole batch) and rd_hits (u32, each
    // query's hits ascending).  The chunks of radius_host run one after the other on one workspace set, so the workspace
    // stays bounded per chunk; only the hits grow with the result.  *total_out = rd_offs[nq].
    int radius_device(const DeviceTree<A>& t, const A* q, size_t nq, size_t stride, A r, cudaStream_t st, uint64_t* total_out,
                      uint32_t* n_chunks_out) {
        const size_t chunk = nq <= (1u << 18) ? std::max<size_t>(nq, 1) : (1u << 17);
        const size_t n_chunks = (nq + chunk - 1) / chunk;
        TRY(rd_offs.ensure((nq + 1) * 8));
        TRY(rd_hits.ensure(4));
        TRY(radius_workspace(t, 1, chunk));
        if (!pin_tot) TRY(pin_tot.create(2 * sizeof(unsigned long long)));
        CU(cudaMemsetAsync(rd_offs.p, 0, 8, st));
        uint64_t total = 0;
        for (size_t c = 0; c < n_chunks; ++c) {
            const size_t q0 = c * chunk;
            const uint32_t cq = (uint32_t)std::min(chunk, nq - q0);
            TRY(radius_count(t, 0, q + q0 * stride, stride, cq, r, st));
            CU(cudaMemcpyAsync(pin_tot.as<unsigned long long>(), r_offsets[0].as<uint64_t>() + cq, 8, cudaMemcpyDeviceToHost, st));
            CU(cudaStreamSynchronize(st));
            const uint64_t ctotal = pin_tot.as<unsigned long long>()[0];
            if ((total + ctotal) * 4 > rd_hits.cap) {
                // sized as radius_host sizes its result; a later, denser chunk grows it, keeping the hits of the earlier ones
                const size_t want = c == 0 ? (size_t)((double)ctotal * 1.12 * (double)nq / cq) + 1024 : rd_hits.cap / 4 + rd_hits.cap / 8;
                DevBuf nb;
                TRY(nb.ensure(std::max<size_t>(total + ctotal, want) * 4));
                if (total) CU(cudaMemcpyAsync(nb.p, rd_hits.p, total * 4, cudaMemcpyDeviceToDevice, st));
                rd_hits = std::move(nb);
            }
            TRY(radius_fill(t, 0, cq, r, ctotal, rd_hits.as<uint32_t>() + total, st));
            rebase_offsets_kernel<<<(cq + 255) / 256, 256, 0, st>>>(r_offsets[0].as<uint64_t>() + 1, cq, 0, total, rd_offs.as<uint64_t>() + q0 + 1);
            CU(cudaGetLastError());
            ++counters.kernel_launches;
            total += ctotal;
        }
        *total_out = total;
        *n_chunks_out = (uint32_t)n_chunks;
        return PN_OK;
    }

    // Two-stage software pipeline over chunks of queries, two workspace sets on two streams:
    //   A(c): H2D queries, pad, count traversal, offsets scan, chunk total -> pinned word
    //   B(c): fill traversal at the offsets, per-query sort, D2H of offsets and hits (widened u32 -> u64 on the host)
    // A(c+1) is enqueued before the host blocks on B(c)'s copies, so the next chunk's traversal runs under the D2H and the
    // host-side widening of this one.
    int radius_host(const void* qv, size_t nq, size_t stride, double rr, uint64_t** offs_out, uint64_t** idx_out) override {
        TRY(check_query_args(qv, nq, stride));
        if (!offs_out || !idx_out) return fail(PN_BAD_ARG, "output pointer is null");
        Call call(*this);
        TRY(call.device());
        // an extension (the reference VP tree has no radius query): answered from the ball partition of the same points
        std::shared_ptr<DeviceTree<A>> comp;
        if (tree->ft.kind != 0) TRY(tree->companion(stream, comp));
        const DeviceTree<A>& t = comp ? *comp : *tree;
        const cudaStream_t st = stream;
        TRY(call.open(st));
        const A r = (A)rr;
        const A* q = (const A*)qv;
        TRY(ensure_io());
        cudaStream_t sx[2] = {s_in, s_out};  // the two pipeline streams (alternate chunks)
        // the result arrays, owned here until they are handed to the caller
        struct Free { void operator()(uint64_t* p) const { free(p); } };
        std::unique_ptr<uint64_t[], Free> offs((uint64_t*)malloc((nq + 1) * 8)), hit_buf;
        if (!offs) return fail(PN_OOM, "malloc offsets");
        // on an error return, copies already queued may still write into offs / hit_buf: the device finishes before
        // they are freed (declared after them, so destroyed first)
        struct SyncOnError { bool armed = true; ~SyncOnError() { if (armed) cudaDeviceSynchronize(); } } sync_on_error;
        offs[0] = 0;
        size_t hit_cap = 0, total = 0;
        const size_t chunk = nq <= (1u << 18) ? std::max<size_t>(nq, 1) : (1u << 17);
        const size_t n_chunks = (nq + chunk - 1) / chunk;
        last_used_tensor = false; last_pruned = false;
        if (!pin_tot) TRY(pin_tot.create(2 * sizeof(unsigned long long)));
        const size_t spitch = std::max<size_t>(stride, t.ft.d) * sizeof(A);
        for (int b = 0; b < (n_chunks > 1 ? 2 : 1); ++b) TRY(r_qraw[b].ensure(chunk * t.ft.d * sizeof(A)));
        TRY(radius_workspace(t, n_chunks > 1 ? 2 : 1, chunk));
        TRY(call.start());
        CU(cudaEventRecord(ev[2], st));
        for (int b = 0; b < 2; ++b) CU(cudaStreamWaitEvent(sx[b], ev[0], 0));
        auto stage_a = [&](size_t c) -> int {
            const int b = (int)(c & 1);
            const size_t q0 = c * chunk;
            const uint32_t cq = (uint32_t)std::min(chunk, nq - q0);
            cudaStream_t s = sx[b];
            CU(cudaMemcpy2DAsync(r_qraw[b].p, t.ft.d * sizeof(A), q + q0 * stride, spitch, t.ft.d * sizeof(A), cq, cudaMemcpyHostToDevice, s));
            TRY(radius_count(t, b, r_qraw[b].as<A>(), t.ft.d, cq, r, s));
            CU(cudaMemcpyAsync(&pin_tot.as<unsigned long long>()[b], r_offsets[b].as<uint64_t>() + cq, 8, cudaMemcpyDeviceToHost, s));
            CU(cudaEventRecord(e_in[b], s));
            counters.h2d_bytes += (uint64_t)cq * t.ft.d * sizeof(A);
            return PN_OK;
        };
        if (n_chunks) TRY(stage_a(0));
        for (size_t c = 0; c < n_chunks; ++c) {
            const int b = (int)(c & 1);
            const size_t q0 = c * chunk;
            const uint32_t cq = (uint32_t)std::min(chunk, nq - q0);
            cudaStream_t s = sx[b];
            if (c + 1 < n_chunks) TRY(stage_a(c + 1));
            CU(cudaEventSynchronize(e_in[b]));
            const uint64_t ctotal = pin_tot.as<unsigned long long>()[b];  // chunk-local total
            if (total + ctotal > hit_cap) {
                // sized once from the first chunk's density (+12 %); grows only if later chunks are denser
                size_t ncap = std::max<size_t>(total + ctotal, c == 0 ? (size_t)((double)ctotal * 1.12 * (double)nq / cq) + 1024 : hit_cap + hit_cap / 2);
                std::unique_ptr<uint64_t[], Free> nb((uint64_t*)result_alloc(ncap * 8));
                if (!nb) return fail(PN_OOM, "allocating the result indices");
                if (hit_buf) memcpy(nb.get(), hit_buf.get(), total * 8);
                hit_buf = std::move(nb); hit_cap = ncap;
            }
            TRY(r_hits[b].ensure((ctotal ? ctotal : 1) * 4));
            TRY(radius_fill(t, b, cq, r, ctotal, r_hits[b].as<uint32_t>(), s));
            CU(cudaMemcpyAsync(offs.get() + q0 + 1, r_offsets[b].as<uint64_t>() + 1, (size_t)cq * 8, cudaMemcpyDeviceToHost, s));
            // the hits, u32 on the device, widened to u64 on up to 12 host threads
            TRY(copy_out_staged(r_hits[b].p, ctotal * 4, s, 12, 4, widen_to(hit_buf.get() + total)));
            CU(cudaStreamSynchronize(s));
            if (total) for (uint32_t i = 1; i <= cq; ++i) offs[q0 + i] += total;  // chunk-local -> global offsets
            total += ctotal;
            counters.d2h_bytes += (uint64_t)cq * 8 + ctotal * 4;
        }
        for (int b = 0; b < 2; ++b) { CU(cudaEventRecord(e_cmp[b], sx[b])); CU(cudaStreamWaitEvent(st, e_cmp[b], 0)); }
        CU(cudaEventRecord(ev[3], st));
        if (!hit_buf) hit_buf.reset((uint64_t*)malloc(8));
        TRY(call.finish(nq));
        sync_on_error.armed = false;
        *offs_out = offs.release();
        *idx_out = hit_buf.release();
        return PN_OK;
    }

    // Radius search from and into device memory (pn_tree_query_radius_dev), enqueued on one stream over the chunks of
    // radius_device: per chunk the count pass scans its offsets onto the total the previous chunk left in offs[q0], and the
    // fill pass writes the hits of the queries that fit below `capacity` straight into the caller's u64 array.  Nothing
    // waits for a result on the host; the workspaces are bounded per chunk.
    int radius_dev(const void* qv, size_t nq, size_t stride, double rr, uint64_t* offs, uint64_t* idx, size_t capacity,
                   cudaStream_t st, bool sync) override {
        TRY(check_query_args(qv, nq, stride));
        if (!offs) return fail(PN_BAD_ARG, "offsets_dev is null");
        if (!idx && capacity) return fail(PN_BAD_ARG, "indices_dev is null with capacity > 0");
        Call call(*this);
        TRY(call.device());
        std::shared_ptr<DeviceTree<A>> comp;   // a VP handle answers from its ball companion, as radius_host does
        if (nq && tree->ft.kind != 0) TRY(tree->companion(stream, comp));
        const DeviceTree<A>& t = comp ? *comp : *tree;
        TRY(call.open(st ? st : (cudaStream_t)stream));
        const A r = (A)rr;
        const A* q = (const A*)qv;
        const size_t chunk = nq <= (1u << 18) ? std::max<size_t>(nq, 1) : (1u << 17);
        last_used_tensor = false; last_pruned = false;
        // every allocation before the first enqueue (a cudaMalloc can synchronise)
        TRY(radius_workspace(t, 1, chunk));
        TRY(r_llist.ensure(chunk * 4));
        TRY(call.start());
        if (nq == 0) CU(cudaMemsetAsync(offs, 0, 8, call.st));
        CU(cudaEventRecord(ev[2], call.st));
        for (size_t q0 = 0; q0 < nq; q0 += chunk) {
            const uint32_t cq = (uint32_t)std::min(chunk, nq - q0);
            TRY(radius_count(t, 0, q + q0 * stride, stride, cq, r, call.st, offs + q0, q0 ? offs + q0 : nullptr));
            TRY(radius_fill<uint64_t>(t, 0, cq, r, 0, idx, call.st, offs + q0, capacity));
        }
        CU(cudaEventRecord(ev[3], call.st));
        return call.finish(nq, sync);
    }

    // ---- point sharding by subtree: local scan -> NCCL exchange -> k-way merge, pipelined over chunks of queries ----------
    int knn_sharded(pn_comm* cm, const void* qv, size_t nq, size_t stride, size_t k, uint32_t exchange, uint64_t* idx_out, void* dist_outv,
                    cudaStream_t st, pn_shard_stats* stats) override {
        TRY(check_query_args(qv, nq, stride));
        if (!cm || !cm->comm) return fail(PN_BAD_ARG, "comm is null");
        if (cm->device != tree->device) return fail(PN_BAD_ARG, "the communicator rank and the tree live on different devices");
        if (k > 255) return fail(PN_BAD_ARG, "sharded k-NN serves k <= 255");
        if (exchange > PN_EXCHANGE_SLICE) return fail(PN_BAD_ARG, "bad exchange mode");
        if (cm->world > 64) return fail(PN_BAD_ARG, "at most 64 ranks");
        if (stats) *stats = pn_shard_stats{};
        if (k == 0 || nq == 0) return PN_OK;
        if (!idx_out || !dist_outv) return fail(PN_BAD_ARG, "output buffer is null");
        Call call(*this);
        if (!st) st = stream;
        TRY(call.open(st));
        TRY(ensure_io());
        const A* q = (const A*)qv;
        A* dist_out = (A*)dist_outv;
        const int W = cm->world, R = cm->rank;
        constexpr bool PACKED = sizeof(A) == 4;
        // chunks of whole waves, about eight of them: the exchange of chunk i hides under the scan of chunk i+1, so only the
        // last chunk's exchange is exposed
        const size_t chunk = shard_chunk(nq), n_chunks = (nq + chunk - 1) / chunk;
        auto slice = [&](int r, size_t& lo, size_t& hi) { pn_query_slice(nq, r, W, &lo, &hi); };
        size_t my_lo = 0, my_hi = nq;
        if (exchange == PN_EXCHANGE_SLICE) slice(R, my_lo, my_hi);
        for (int b = 0; b < (n_chunks > 1 ? 2 : 1); ++b) {
            TRY(sh_li[b].ensure(chunk * k * 8));
            TRY(sh_ld[b].ensure(chunk * k * sizeof(A)));
            TRY(sh_gat[b].ensure((size_t)W * chunk * k * 8));
            if (PACKED) TRY(sh_pack[b].ensure(chunk * k * 8)); else TRY(sh_gat_d[b].ensure((size_t)W * chunk * k * sizeof(A)));
        }
        TRY(grow_events(sh_ev, 6 * n_chunks, cudaEventDefault));
        auto EV = [&](size_t c, int i) -> cudaEvent_t { return sh_ev[6 * c + i]; };  // 0,1 scan; 2,3 exchange; 4,5 merge
        cudaStream_t cs = cm->stream;
        TRY(call.start());
        unsigned long long bytes = 0, calls = 0, rows_out = 0;
        // rows of chunk [c0, c1) owned by rank r (SLICE) / all of them (ALLGATHER)
        auto owned = [&](int r, size_t c0, size_t c1, size_t& lo, size_t& cnt) {
            size_t slo = 0, shi = nq;
            if (exchange == PN_EXCHANGE_SLICE) slice(r, slo, shi);
            lo = std::max(c0, slo);
            const size_t hi = std::min(c1, shi);
            cnt = hi > lo ? hi - lo : 0;
        };
        auto merge_chunk = [&](size_t c) -> int {
            const int b = (int)(c & 1);
            const size_t c0 = c * chunk, c1 = std::min(nq, c0 + chunk);
            size_t lo, cnt;
            owned(R, c0, c1, lo, cnt);
            CU(cudaStreamWaitEvent(st, EV(c, 3), 0));
            CU(cudaEventRecord(EV(c, 4), st));
            if (cnt) {
                const size_t orow = lo - my_lo;
                if constexpr (PACKED) {
                    merge_packed_kernel<<<(unsigned)((cnt + 127) / 128), 128, 0, st>>>(sh_gat[b].as<unsigned long long>(), (uint32_t)W, cnt * k, (uint32_t)cnt,
                                                                                       (uint32_t)k, idx_out + orow * k, (float*)dist_out + orow * k);
                } else {
                    CU(merge_lists<A, uint64_t>(st, sh_gat_d[b].as<A>(), sh_gat[b].as<uint64_t>(), (uint32_t)W,
                                                                                                  (uint32_t)cnt, (uint32_t)k, idx_out + orow * k,
                                                                                                  dist_out + orow * k, (uint32_t)k, 0, nullptr, nullptr));
                }
                CU(cudaGetLastError());
                ++counters.kernel_launches;
                rows_out += cnt;
            }
            CU(cudaEventRecord(EV(c, 5), st));
            return PN_OK;
        };
        for (size_t c = 0; c < n_chunks; ++c) {
            const int b = (int)(c & 1);
            const size_t c0 = c * chunk, c1 = std::min(nq, c0 + chunk);
            const uint32_t cq = (uint32_t)(c1 - c0);
            // scan: the local lists of chunk c (the buffers of chunk c-2 have been sent: the exchange of c-2 is awaited)
            if (c >= 2) CU(cudaStreamWaitEvent(st, EV(c - 2, 3), 0));
            CU(cudaEventRecord(EV(c, 0), st));
            TRY(knn_device(*tree, q + c0 * stride, cq, stride, (uint32_t)k, sh_li[b].as<uint64_t>(), sh_ld[b].as<A>(), st));
            if constexpr (PACKED) {
                const size_t cnt = (size_t)cq * k;
                pack_lists_kernel<<<(unsigned)((cnt + 255) / 256), 256, 0, st>>>(sh_li[b].as<uint64_t>(), (const float*)sh_ld[b].p, cnt,
                                                                                 sh_pack[b].as<unsigned long long>());
                CU(cudaGetLastError());
                ++counters.kernel_launches;
            }
            CU(cudaEventRecord(EV(c, 1), st));
            // exchange on the communicator's stream: runs under the scan of chunk c+1 (the gather buffer of chunk c-2 must
            // have been merged)
            CU(cudaStreamWaitEvent(cs, EV(c, 1), 0));
            if (c >= 2) CU(cudaStreamWaitEvent(cs, EV(c - 2, 5), 0));
            CU(cudaEventRecord(EV(c, 2), cs));
            if (exchange == PN_EXCHANGE_ALLGATHER) {
                if constexpr (PACKED) {
                    NC(cm->api->AllGather(sh_pack[b].p, sh_gat[b].p, (size_t)cq * k, ncclUint64, cm->comm, cs));
                    bytes += (unsigned long long)(W - 1) * cq * k * 8; ++calls;
                } else {
                    NC(cm->api->GroupStart());
                    NC(cm->api->AllGather(sh_li[b].p, sh_gat[b].p, (size_t)cq * k, ncclUint64, cm->comm, cs));
                    NC(cm->api->AllGather(sh_ld[b].p, sh_gat_d[b].p, (size_t)cq * k, ncclFloat64, cm->comm, cs));
                    NC(cm->api->GroupEnd());
                    bytes += (unsigned long long)(W - 1) * cq * k * 16; calls += 2;
                }
            } else {
                size_t mlo, mcnt;
                owned(R, c0, c1, mlo, mcnt);
                NC(cm->api->GroupStart());
                for (int p = 0; p < W; ++p) {
                    size_t plo, pcnt;
                    owned(p, c0, c1, plo, pcnt);
                    if (pcnt) {  // rows of this chunk that rank p merges: my lists for them go to p
                        const size_t off = (plo - c0) * k;
                        if constexpr (PACKED) {
                            NC(cm->api->Send(sh_pack[b].as<unsigned long long>() + off, pcnt * k, ncclUint64, p, cm->comm, cs));
                        } else {
                            NC(cm->api->Send(sh_li[b].as<uint64_t>() + off, pcnt * k, ncclUint64, p, cm->comm, cs));
                            NC(cm->api->Send(sh_ld[b].as<A>() + off, pcnt * k, ncclFloat64, p, cm->comm, cs));
                        }
                        if (p != R) bytes += (unsigned long long)pcnt * k * (PACKED ? 8 : 16);
                        calls += PACKED ? 1 : 2;
                    }
                    if (mcnt) {  // and every rank's lists for my rows arrive here, list p at [p][mcnt][k]
                        if constexpr (PACKED) {
                            NC(cm->api->Recv(sh_gat[b].as<unsigned long long>() + (size_t)p * mcnt * k, mcnt * k, ncclUint64, p, cm->comm, cs));
                        } else {
                            NC(cm->api->Recv(sh_gat[b].as<uint64_t>() + (size_t)p * mcnt * k, mcnt * k, ncclUint64, p, cm->comm, cs));
                            NC(cm->api->Recv(sh_gat_d[b].as<A>() + (size_t)p * mcnt * k, mcnt * k, ncclFloat64, p, cm->comm, cs));
                        }
                    }
                }
                NC(cm->api->GroupEnd());
            }
            CU(cudaEventRecord(EV(c, 3), cs));
            if (c >= 1) TRY(merge_chunk(c - 1));   // after the scan of chunk c is queued, so the exchange of c-1 had time to run
        }
        TRY(merge_chunk(n_chunks - 1));
        TRY(call.finish(nq));
        cm->bytes_sent += bytes; cm->collectives += calls;
        if (stats) {
            float ms = 0.f;
            for (size_t c = 0; c < n_chunks; ++c) {
                if (cudaEventElapsedTime(&ms, EV(c, 0), EV(c, 1)) == cudaSuccess) stats->scan_ms += ms;
                if (cudaEventElapsedTime(&ms, EV(c, 2), EV(c, 3)) == cudaSuccess) stats->exchange_ms += ms;
                if (cudaEventElapsedTime(&ms, EV(c, 4), EV(c, 5)) == cudaSuccess) stats->merge_ms += ms;
            }
            if (cudaEventElapsedTime(&ms, ev[0], ev[1]) == cudaSuccess) stats->total_ms = ms;
            (void)cudaGetLastError();
            stats->nccl_bytes_sent = bytes; stats->nccl_calls = calls; stats->rows_out = rows_out; stats->n_chunks = (uint32_t)n_chunks;
        }
        return PN_OK;
    }

    // whole waves per chunk, about eight chunks (see knn_sharded)
    size_t shard_chunk(size_t nq) const override {
        const size_t wave = (size_t)n_sms * tree->query_tile();
        return nq < 2 * wave ? nq : std::min<size_t>(std::max<size_t>(1, (nq / 8 + wave - 1) / wave) * wave, ((size_t)1 << 20) / wave * wave);
    }
    // ---- point sharding by subtree WITHOUT a collective (one process, several GPUs): the merge kernel of every rank reads
    // the other ranks' packed lists straight from their memory over NVLink.  Every rank scans chunk after chunk on its own
    // stream into ONE packed buffer covering all queries (8 k bytes per query), recording an event per chunk; after the
    // rank threads have met once (an event must be recorded before another device's stream can wait on it), the merges of
    // all chunks are queued on a second stream, each waiting for that chunk's events of every rank.  No rank's scan ever
    // waits for another rank.
    int knn_sharded_peer(PeerShared& ps, int R, int W, const void* qv, size_t nq, size_t stride, size_t k, uint64_t* idx_out, void* dist_outv,
                         pn_shard_stats* stats) override {
        if constexpr (sizeof(A) != 4) {
            (void)ps; (void)R; (void)W; (void)qv; (void)nq; (void)stride; (void)k; (void)idx_out; (void)dist_outv; (void)stats;
            return fail(PN_BAD_ARG, "the peer exchange serves f32 trees");
        } else {
            struct Guard { PeerShared& p; bool ok = false; ~Guard() { if (!ok) p.fail(); } } guard{ps};
            TRY(check_query_args(qv, nq, stride));
            if (k == 0 || k > 255 || W > 64) return fail(PN_BAD_ARG, "peer exchange: 1 <= k <= 255, at most 64 ranks");
            Call call(*this);
            const cudaStream_t st = stream;
            TRY(call.open(st));
            TRY(ensure_io());
            cudaStream_t ms = s_out;   // the merge stream
            if (stats) *stats = pn_shard_stats{};
            const A* q = (const A*)qv;
            const size_t chunk = ps.chunk, n_chunks = ps.n_chunks;
            size_t my_lo, my_hi;
            pn_query_slice(nq, R, W, &my_lo, &my_hi);
            DevBuf& ptrs = sh_gat[0];    // [W] list pointers of every rank
            DevBuf& packall = sh_gat[1]; // this rank's packed lists of all queries
            TRY(ptrs.ensure((size_t)W * sizeof(void*)));
            TRY(packall.ensure(nq * k * 8));
            for (int b = 0; b < 2; ++b) {
                TRY(sh_li[b].ensure(chunk * k * 8));
                TRY(sh_ld[b].ensure(chunk * k * 4));
            }
            ps.pack[R] = packall.as<unsigned long long>();
            TRY(grow_events(sh_ev, 2 * n_chunks + 2, cudaEventDefault));
            auto EV = [&](size_t c, int i) -> cudaEvent_t { return sh_ev[2 * c + i]; };  // scan start / end of chunk c; the last two: merge start / end
            TRY(call.start());
            for (size_t c = 0; c < n_chunks; ++c) {
                const int b = (int)(c & 1);
                const size_t c0 = c * chunk, c1 = std::min(nq, c0 + chunk);
                const uint32_t cq = (uint32_t)(c1 - c0);
                CU(cudaEventRecord(EV(c, 0), st));
                TRY(knn_device(*tree, q + c0 * stride, cq, stride, (uint32_t)k, sh_li[b].as<uint64_t>(), sh_ld[b].as<A>(), st));
                const size_t cnt = (size_t)cq * k;
                pack_lists_kernel<<<(unsigned)((cnt + 255) / 256), 256, 0, st>>>(sh_li[b].as<uint64_t>(), (const float*)sh_ld[b].p, cnt,
                                                                                 packall.as<unsigned long long>() + c0 * k);
                CU(cudaGetLastError());
                ++counters.kernel_launches;
                CU(cudaEventRecord(EV(c, 1), st));
                CU(cudaEventRecord(ps.ev_scan[R][c], st));
            }
            if (!ps.barrier()) return ps.released();   // every rank's buffers exist and all scan events are recorded
            std::vector<const unsigned long long*> hp(ps.pack.begin(), ps.pack.end());
            CU(cudaMemcpyAsync(ptrs.p, hp.data(), hp.size() * sizeof(void*), cudaMemcpyHostToDevice, ms));
            unsigned long long rows_out = 0, peer_bytes = 0;
            CU(cudaEventRecord(EV(n_chunks, 0), ms));
            for (size_t c = 0; c < n_chunks; ++c) {
                const size_t c0 = c * chunk, c1 = std::min(nq, c0 + chunk);
                const size_t lo = std::max(c0, my_lo), hi = std::min(c1, my_hi);
                if (hi <= lo) continue;
                for (int p = 0; p < W; ++p) CU(cudaStreamWaitEvent(ms, ps.ev_scan[p][c], 0));   // every rank's lists of chunk c are packed
                const size_t cnt = hi - lo;
                merge_packed_peer_kernel<<<(unsigned)((cnt + 127) / 128), 128, 0, ms>>>(
                    reinterpret_cast<const unsigned long long* const*>(ptrs.p), (uint32_t)W, lo, (uint32_t)cnt, (uint32_t)k,
                    idx_out + (lo - my_lo) * k, (float*)dist_outv + (lo - my_lo) * k);
                CU(cudaGetLastError());
                ++counters.kernel_launches;
                rows_out += cnt;
                peer_bytes += (unsigned long long)(W - 1) * cnt * k * 8;
            }
            CU(cudaEventRecord(EV(n_chunks, 1), ms));
            CU(cudaStreamWaitEvent(st, EV(n_chunks, 1), 0));
            CU(cudaEventRecord(ev[1], st));
            CU(cudaStreamSynchronize(st));
            // nobody may free or reuse a packed buffer while a peer still reads it
            if (!ps.barrier()) return ps.released();
            guard.ok = true;
            if (stats) {
                float ms_ = 0.f;
                for (size_t c = 0; c < n_chunks; ++c)
                    if (cudaEventElapsedTime(&ms_, EV(c, 0), EV(c, 1)) == cudaSuccess) stats->scan_ms += ms_;
                // exposed tail: end of this rank's last scan to the end of its last merge (waits for the slowest rank included)
                if (cudaEventElapsedTime(&ms_, EV(n_chunks - 1, 1), EV(n_chunks, 1)) == cudaSuccess) stats->merge_ms = ms_;
                if (cudaEventElapsedTime(&ms_, ev[0], ev[1]) == cudaSuccess) stats->total_ms = ms_;
                (void)cudaGetLastError();
                stats->nccl_bytes_sent = 0; stats->nccl_calls = 0; stats->rows_out = rows_out; stats->n_chunks = (uint32_t)n_chunks;
                stats->peer_mib = (uint32_t)std::min<unsigned long long>((peer_bytes + (1u << 20) - 1) >> 20, 0xffffffffull);
            }
            return fetch_counters(st, nq);
        }
    }

    // ---- radius search of a multi-GPU handle (pn_multi_balltree_query_radius_f32), called on every rank's thread.  `q` holds
    // the caller's nq host queries; rank R owns result rows [lo, hi) = pn_query_slice(nq, R, W).
    //   REPLICATE: radius_device over the slice on this rank's replica.
    //   BY_SUBTREE: radius_device over ALL queries on this rank's shard; once the ranks have met, the owner of a slice pulls
    //   every shard's offsets and hits of that slice into local staging (cudaMemcpyPeerAsync: over NVLink with peer access,
    //   staged by the driver without it; no collective, so pn_multi_set_exchange does not apply) and merges the lists by
    //   rank (merge_radius_lists, u32).  Shard trees hold global ids, so the hits need no translation.
    // Then every rank publishes its slice total; rank 0 allocates the single result once all totals are known, and every
    // rank writes its offsets (plus the totals of the slices before it) and its hits, widened to u64, into its region.
    int radius_multi(PeerShared& ps, int R, int W, bool by_subtree, const void* qv, size_t nq, size_t stride, double rr,
                     pn_shard_stats* stats) override {
        if constexpr (sizeof(A) != 4) {
            (void)ps; (void)R; (void)W; (void)by_subtree; (void)qv; (void)nq; (void)stride; (void)rr; (void)stats;
            return fail(PN_BAD_ARG, "multi-GPU radius search serves f32 trees");
        } else {
            struct Guard { PeerShared& p; bool ok = false; ~Guard() { if (!ok) p.fail(); } } guard{ps};
            TRY(check_query_args(qv, nq, stride));
            if (stats) *stats = pn_shard_stats{};
            size_t lo, hi;
            pn_query_slice(nq, R, W, &lo, &hi);
            const size_t rows = hi - lo, nql = by_subtree ? nq : rows;   // rows owned, queries traversed
            const size_t d = tree->ft.d;
            Call call(*this);
            const cudaStream_t st = stream;
            TRY(call.open(st));
            // on an error return, a copy into the caller's result may still be queued: the device finishes before the
            // result is freed (declared after `guard` and `call`, so destroyed first)
            struct SyncOnError { bool armed = true; ~SyncOnError() { if (armed) cudaDeviceSynchronize(); } } sync_on_error;
            last_used_tensor = false; last_pruned = false;
            TRY(rd_q.ensure(std::max<size_t>(nql, 1) * d * 4));
            TRY(grow_events(sh_ev, 5, cudaEventDefault));   // traversal start / end, pulls end, merge end, pulls start
            TRY(call.start());
            if (nql) {
                const float* q = (const float*)qv + (by_subtree ? 0 : lo * stride);
                CU(cudaMemcpy2DAsync(rd_q.p, d * 4, q, std::max(stride, d) * 4, d * 4, nql, cudaMemcpyHostToDevice, st));
            }
            counters.h2d_bytes = (uint64_t)nql * d * 4;
            CU(cudaEventRecord(sh_ev[0], st));
            uint64_t slice_total = 0;
            uint32_t n_chunks = 0;
            TRY(radius_device(*tree, rd_q.as<float>(), nql, d, (float)rr, st, &slice_total, &n_chunks));
            CU(cudaEventRecord(sh_ev[1], st));
            const uint64_t* offs_dev = rd_offs.as<uint64_t>();   // this rank's slice as CSR on the device
            const uint32_t* hits_dev = rd_hits.as<uint32_t>();
            unsigned long long peer_bytes = 0;
            const bool pulled = by_subtree && rows;
            if (by_subtree) {
                std::vector<uint64_t>& bnd = ps.r_bound[R];   // this shard's offsets at every rank's slice start, and at nq
                bnd.assign(W + 1, 0);
                for (int j = 0; j <= W; ++j) {
                    size_t b = nq;
                    if (j < W) pn_query_slice(nq, j, W, &b, nullptr);
                    CU(cudaMemcpyAsync(&bnd[j], rd_offs.as<uint64_t>() + b, 8, cudaMemcpyDeviceToHost, st));
                }
                CU(cudaStreamSynchronize(st));
                ps.r_offs[R] = rd_offs.as<uint64_t>();
                ps.r_hits[R] = rd_hits.as<uint32_t>();
                ps.r_dev[R] = tree->device;
                if (!ps.barrier()) return ps.released();   // every shard's CSR is complete
                std::vector<uint64_t> base(W + 1, 0);   // where shard s's hits of this slice start in the pulled staging
                for (int s = 0; s < W; ++s) base[s + 1] = base[s] + (ps.r_bound[s][R + 1] - ps.r_bound[s][R]);
                slice_total = base[W];
                if (pulled) {
                    TRY(rp_offs.ensure((size_t)W * (rows + 1) * 8));
                    TRY(rp_hits.ensure(std::max<uint64_t>(slice_total, 1) * 4));
                    TRY(rm_offs.ensure((rows + 1) * 8));
                    TRY(rm_hits.ensure(std::max<uint64_t>(slice_total, 1) * 4));
                    TRY(r_counts[0].ensure(rows * 4));
                    TRY(r_sums[0].ensure((rows / SCAN_BLOCK + 1) * 8));
                    uint64_t* po = rp_offs.as<uint64_t>();
                    CU(cudaEventRecord(sh_ev[4], st));
                    for (int s = 0; s < W; ++s) {
                        const uint64_t nh = base[s + 1] - base[s];
                        CU(cudaMemcpyPeerAsync(po + (size_t)s * (rows + 1), tree->device, ps.r_offs[s] + lo, ps.r_dev[s], (rows + 1) * 8, st));
                        if (nh) CU(cudaMemcpyPeerAsync(rp_hits.as<uint32_t>() + base[s], tree->device, ps.r_hits[s] + ps.r_bound[s][R], ps.r_dev[s], nh * 4, st));
                        if (s != R) peer_bytes += (rows + 1) * 8 + nh * 4;
                    }
                    CU(cudaEventRecord(sh_ev[2], st));
                    // shard s's offsets into its own hit array -> positions in the concatenation of the pulled hits
                    for (int s = 0; s < W; ++s)
                        rebase_offsets_kernel<<<(unsigned)((rows + 1 + 255) / 256), 256, 0, st>>>(po + (size_t)s * (rows + 1), rows + 1, ps.r_bound[s][R],
                                                                                                 base[s], po + (size_t)s * (rows + 1));
                    const unsigned blocks = (unsigned)std::max<uint64_t>(1, std::min<uint64_t>((slice_total + 255) / 256, 8ull * n_sms));
                    CU(merge_radius_lists<uint32_t>(st, po, rp_hits.as<uint32_t>(), (uint32_t)W, (uint32_t)rows, rm_offs.as<uint64_t>(),
                                                    rm_hits.as<uint32_t>(), r_counts[0].as<uint32_t>(), r_sums[0].as<unsigned long long>(), blocks));
                    CU(cudaEventRecord(sh_ev[3], st));
                    counters.kernel_launches += (uint64_t)W + 4;
                    offs_dev = rm_offs.as<uint64_t>();
                    hits_dev = rm_hits.as<uint32_t>();
                }
                // the pulls are done before this rank passes the next barrier, so no rank reads another's buffers after it
                CU(cudaStreamSynchronize(st));
            }
            ps.r_total[R] = slice_total;
            if (!ps.barrier()) return ps.released();   // every slice total is known
            if (R == 0) {
                uint64_t all = 0;
                for (uint64_t t : ps.r_total) all += t;
                ps.r_out_offs = (uint64_t*)result_alloc((nq + 1) * 8);
                ps.r_out_hits = (uint64_t*)result_alloc(all * 8);
                if (!ps.r_out_offs || !ps.r_out_hits) return fail(PN_OOM, "allocating the result");
                ps.r_out_offs[0] = 0;
            }
            if (!ps.barrier()) return ps.released();   // the result is allocated
            if (rows) {
                uint64_t base = 0;
                for (int j = 0; j < R; ++j) base += ps.r_total[j];
                uint64_t* offs_out = ps.r_out_offs + lo;
                CU(cudaMemcpyAsync(offs_out + 1, offs_dev + 1, rows * 8, cudaMemcpyDeviceToHost, st));
                TRY(copy_out_staged(hits_dev, slice_total * 4, st, 12, 4, widen_to(ps.r_out_hits + base)));
                CU(cudaStreamSynchronize(st));
                if (base) for (size_t i = 1; i <= rows; ++i) offs_out[i] += base;
            }
            counters.d2h_bytes = (uint64_t)rows * 8 + slice_total * 4;
            TRY(call.finish(nql));
            sync_on_error.armed = false;
            guard.ok = true;
            if (stats) {
                float ms = 0.f;
                if (cudaEventElapsedTime(&ms, sh_ev[0], sh_ev[1]) == cudaSuccess) stats->scan_ms = ms;
                if (pulled && cudaEventElapsedTime(&ms, sh_ev[4], sh_ev[2]) == cudaSuccess) stats->exchange_ms = ms;
                if (pulled && cudaEventElapsedTime(&ms, sh_ev[2], sh_ev[3]) == cudaSuccess) stats->merge_ms = ms;
                (void)cudaGetLastError();
                stats->total_ms = counters.device_ms;
                stats->rows_out = rows; stats->n_chunks = n_chunks;
                stats->peer_mib = (uint32_t)std::min<unsigned long long>((peer_bytes + (1u << 20) - 1) >> 20, 0xffffffffull);
            }
            return PN_OK;
        }
    }

    int replicate_send(pn_comm* cm, int root) override {
        if (host_only) return fail(PN_BAD_ARG, "a host-only tree has nothing to replicate");
        if (cm->device != tree->device) return fail(PN_BAD_ARG, "the communicator rank and the tree live on different devices");
        Call call(*this);
        TRY(call.device());
        return tree->replicate_send(cm, root);
    }

    // ---- sessions: a second handle onto the same tree (pn_tree_session).  The tree is shared; everything a call writes
    // (stream, events, workspaces, counters, the mutex) is the session's own, so calls on different sessions of one tree
    // overlap on the device.
    int session(pn_tree** out) override {
        if (host_only) return fail(PN_BAD_ARG, "a host-only tree has no device arrays to share");
        std::unique_ptr<Engine> e;
        TRY(open(tree, false, e));
        e->info = info;
        e->owns_tree = false;
        *out = e.release();
        return PN_OK;
    }

    int layout(uint32_t* ids, uint32_t* blo, uint32_t* bhi, void* rad, void* cen, void* pts) override {
        const DeviceTree<A>& t = *tree;
        if (t.gpu_built) {
            DeviceGuard g(t.device);
            if (ids) CU(cudaMemcpy(ids, t.d_ids.p, (size_t)t.ft.n * 4, cudaMemcpyDeviceToHost));
            if (rad) CU(cudaMemcpy(rad, t.d_radii.p, (size_t)t.ft.n_nodes * sizeof(A), cudaMemcpyDeviceToHost));
            if (cen) CU(cudaMemcpy(cen, t.d_centers.p, (size_t)t.ft.n_nodes * t.ft.dpad * sizeof(A), cudaMemcpyDeviceToHost));
            ids = nullptr; rad = nullptr; cen = nullptr;
        }
        if (ids) memcpy(ids, t.ft.ids.data(), t.ft.ids.size() * 4);
        if (blo) memcpy(blo, t.ft.bucket_lo.data(), t.ft.bucket_lo.size() * 4);
        if (bhi) memcpy(bhi, t.ft.bucket_hi.data(), t.ft.bucket_hi.size() * 4);
        if (rad) memcpy(rad, t.ft.radii.data(), (size_t)t.ft.n_nodes * sizeof(A));
        if (cen) memcpy(cen, t.ft.centers.data(), (size_t)t.ft.n_nodes * t.ft.dpad * sizeof(A));
        if (pts) {
            if (host_only) memcpy(pts, t.ft.pts.data(), t.ft.pts.size() * sizeof(A));
            else {
                DeviceGuard g(t.device);
                CU(cudaMemcpy(pts, t.d_pts.p, (size_t)t.ft.n * t.ft.dpad * sizeof(A), cudaMemcpyDeviceToHost));
            }
        }
        return PN_OK;
    }
};
#undef NC

template <typename A>
static int finish_create(int kind, std::unique_ptr<Engine<A>>& e, const pn_build_opts& o, std::chrono::steady_clock::time_point t0, pn_tree** out);

// The caller's build options, as far as its struct_size reaches (none: the defaults on the current device), with the
// bucket size normalised.
static pn_build_opts read_build_opts(const pn_build_opts* in) {
    pn_build_opts o{};
    if (in) memcpy(&o, in, std::min<size_t>(sizeof(o), in->struct_size ? in->struct_size : sizeof(o)));
    else o.device = -1;
    o.bucket_size = o.bucket_size ? std::max(o.bucket_size, 8u) : 256;
    return o;
}
// the checks every tree build makes, after those of its entry point
static int check_build_opts(const pn_build_opts& o, int kind) {
    if (o.prune > PN_PRUNE_OFF) return fail(PN_BAD_ARG, "bad prune option");
    if (o.partition > PN_PARTITION_TWO_MEANS) return fail(PN_BAD_ARG, "bad partition option");
    if (o.shard_depth && (kind != PN_KIND_BALL || o.shard_depth > 16 || o.shard_index >= (1u << o.shard_depth)))
        return fail(PN_BAD_ARG, kind != PN_KIND_BALL ? "subtree sharding is a ball-tree option" : "bad shard_depth / shard_index");
    return PN_OK;
}
// A new handle with an empty tree on the device of `o` (-1: the current one) for the build to fill
template <typename A>
static int new_tree_handle(const pn_build_opts& o, bool host_only, std::unique_ptr<Engine<A>>& e) {
    int dev = o.device;
    if (!host_only && dev < 0 && cudaGetDevice(&dev) != cudaSuccess) {
        (void)cudaGetLastError();
        return fail(PN_CUDA, "no CUDA device available (there is no CPU fallback)");
    }
    auto t = std::make_shared<DeviceTree<A>>();
    t->device = dev;
    t->algo = o.algo;
    t->prune_opt = o.prune;
    return Engine<A>::open(std::move(t), host_only, e);
}

template <typename A>
static int create_tree(int kind, const A* points, size_t n, size_t d, size_t row_stride, size_t col_stride,
                       const pn_build_opts* opts_in, pn_tree** out) {
    if (!out) return fail(PN_BAD_ARG, "out is null");
    *out = nullptr;
    if (n == 0) return fail(PN_EMPTY, "array is empty");                                         // src/ball_tree.rs:44-46
    if (d > 1 && col_stride != 1) return fail(PN_NOT_CONTIGUOUS, "array is not contiguous in memory");  // :47-49
    if (!points) return fail(PN_BAD_ARG, "points is null");
    if (d == 0) return fail(PN_BAD_ARG, "points have zero columns");
    if (n >= 0xFFFFFFFFull) return fail(PN_BAD_ARG, "n must be < 2^32 - 1 (u32 indices inside the engine)");
    if (n > 1 && row_stride < d) return fail(PN_BAD_ARG, "row_stride < dimension");
    const pn_build_opts o = read_build_opts(opts_in);
    const uint32_t bucket = o.bucket_size;
    uint32_t threads = o.host_threads ? o.host_threads : std::max(1u, std::thread::hardware_concurrency());
    auto t0 = std::chrono::steady_clock::now();
    std::unique_ptr<Engine<A>> e;
    const bool host_only = (o.flags & PN_FLAG_HOST_ONLY) != 0;
    if (o.builder > PN_BUILDER_DEVICE) return fail(PN_BAD_ARG, "bad builder");
    TRY(check_build_opts(o, kind));
    // ball trees with a device are built there from 32768 points up (bit-identical layout, tests/test_gpu_build.py)
    const bool on_device = !host_only && (o.builder == PN_BUILDER_DEVICE || (o.builder == PN_BUILDER_AUTO && n >= 32768));
    if (o.builder == PN_BUILDER_DEVICE && !on_device) return fail(PN_BAD_ARG, "the device builder needs a device");
    try {
        TRY(new_tree_handle(o, host_only, e));
        DeviceTree<A>& t = *e->tree;
        if (on_device) {
            // raw rows to the device (dense n x d), partition and flatten there
            DeviceGuard g(t.device);
            if (!g.ok) return fail(PN_CUDA, "no usable CUDA device (there is no CPU fallback)");
            DevBuf raw;
            TRY(raw.ensure(n * d * sizeof(A)));
            cudaError_t ce = cudaMemcpy2D(raw.p, d * sizeof(A), points, std::max(row_stride, d) * sizeof(A), d * sizeof(A), n, cudaMemcpyHostToDevice);
            if (ce != cudaSuccess) return fail(PN_CUDA, std::string("uploading the points: ") + cudaGetErrorString(ce));
            TRY(kind == PN_KIND_BALL ? t.build_on_device(raw.as<A>(), n, d, d, bucket, o.shard_depth, o.shard_index, 0, e->stream)
                                     : t.build_vp_on_device(raw.as<A>(), n, d, d, bucket, e->stream));
        } else if (kind == PN_KIND_BALL) {
            BallBuilder<A> b(points, n, d, row_stride, threads);
            std::vector<uint32_t> idx(n);
            for (size_t i = 0; i < n; ++i) idx[i] = (uint32_t)i;
            size_t lo = 0, hi = n;
            if (o.shard_depth) {
                b.shard_range(idx, o.shard_depth, o.shard_index, lo, hi);
                if (hi == lo) return fail(PN_EMPTY, "shard holds no points");
            }
            b.build(idx, lo, hi, bucket, t.ft);
        } else {
            VpBuilder<A> b(points, n, d, row_stride, threads);
            b.build(bucket, t.ft);
        }
    } catch (const std::bad_alloc&) {
        return fail(PN_OOM, "host allocation failed while building the tree");
    }
    DeviceTree<A>& t = *e->tree;
    if (!host_only && !on_device) TRY(t.upload(e->stream));
    if (kind == PN_KIND_VP && !host_only && t.tensor_ready && n >= 1024) {
        // the ball partition of the same points for the tensor path (see DeviceTree::part); a failure here only loses the speed-up
        DeviceGuard g(t.device);
        DevBuf raw;
        std::shared_ptr<DeviceTree<A>> ball;
        if (g.ok && raw.ensure(n * d * sizeof(A)) == PN_OK &&
            cudaMemcpy2D(raw.p, d * sizeof(A), points, std::max(row_stride, d) * sizeof(A), d * sizeof(A), n, cudaMemcpyHostToDevice) == cudaSuccess &&
            t.build_partition(raw.as<A>(), d, bucket, 0, e->stream, ball) == PN_OK && ball->tensor_ready) {
            raw.release();
            // clustered points: the two-means partition of the same rows instead, when its tile bounds are the tighter ones
            std::shared_ptr<DeviceTree<A>> tm;
            ball->two_means_partition(o.partition, bucket, e->stream, tm);
            t.part = tm ? tm : ball;
        }
        (void)cudaGetLastError();
    }
    if (kind == PN_KIND_BALL && !host_only && !o.shard_depth) t.two_means_partition(o.partition, bucket, e->stream, t.part);
    return finish_create(kind, e, o, t0, out);
}

template <typename A>
static int finish_create(int kind, std::unique_ptr<Engine<A>>& e, const pn_build_opts& o, std::chrono::steady_clock::time_point t0, pn_tree** out) {
    const DeviceTree<A>& t = *e->tree;
    const FlatTree<A>& ft = t.ft;
    pn_tree_info& inf = e->info;
    inf.n_points = ft.n; inf.n_points_total = ft.n_total;
    inf.dim = ft.d; inf.dim_padded = ft.dpad;
    inf.kind = kind; inf.dtype = sizeof(A) == 4 ? PN_F32 : PN_F64;
    inf.n_levels = ft.L; inf.n_buckets = ft.n_buckets; inf.n_nodes = ft.n_nodes;
    inf.bucket_size_max = ft.bucket_max;
    inf.algo = o.algo;
    inf.device = e->host_only ? -1 : t.device;
    {
        const DeviceTree<A>* pe = t.part ? t.part.get() : &t;   // a VP handle reports the ball partition its tensor path uses
        inf.prune_seeded = pe->prune_on ? 1u : 0u; inf.prune_tiles = pe->tiles_on ? 1u : 0u;
        inf.est_seed_candidates = pe->seed_candidates; inf.est_tile_frac = pe->tile_frac; inf.est_group_tile_frac = pe->prune_frac;
        inf.tensor_partition = pe->partition_rule;
    }
    inf.build_seconds = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
    *out = e.release();
    return PN_OK;
}

// points already on the device: BallTree::new with the partition computed there
template <typename A>
static int create_tree_dev(const A* points_dev, size_t n, size_t d, size_t row_stride, const pn_build_opts* opts_in, pn_tree** out) {
    if (!out) return fail(PN_BAD_ARG, "out is null");
    *out = nullptr;
    if (n == 0) return fail(PN_EMPTY, "array is empty");
    if (!points_dev) return fail(PN_BAD_ARG, "points is null");
    if (d == 0) return fail(PN_BAD_ARG, "points have zero columns");
    if (n >= 0xFFFFFFFFull) return fail(PN_BAD_ARG, "n must be < 2^32 - 1 (u32 indices inside the engine)");
    if (n > 1 && row_stride < d) return fail(PN_BAD_ARG, "row_stride < dimension");
    const pn_build_opts o = read_build_opts(opts_in);
    if (o.flags & PN_FLAG_HOST_ONLY) return fail(PN_BAD_ARG, "device-resident points cannot build a host-only tree");
    if (o.builder == PN_BUILDER_HOST) return fail(PN_BAD_ARG, "device-resident points are built on the device");
    TRY(check_build_opts(o, PN_KIND_BALL));
    auto t0 = std::chrono::steady_clock::now();
    std::unique_ptr<Engine<A>> e;
    try {
        TRY(new_tree_handle(o, false, e));
        DeviceTree<A>& t = *e->tree;
        TRY(t.build_on_device(points_dev, n, d, row_stride, o.bucket_size, o.shard_depth, o.shard_index, 0, e->stream));
        if (!o.shard_depth) t.two_means_partition(o.partition, o.bucket_size, e->stream, t.part);
    } catch (const std::bad_alloc&) {
        return fail(PN_OOM, "host allocation failed while building the tree");
    }
    return finish_create(PN_KIND_BALL, e, o, t0, out);
}

// the receiving side of pn_tree_replicate: a new handle onto the broadcast tree
template <typename A>
static int receive_replica(pn_comm* cm, int root, int kind, pn_tree** out) {
    auto t0 = std::chrono::steady_clock::now();
    auto t = std::make_shared<DeviceTree<A>>();
    TRY(t->replicate_recv(cm, root));
    std::unique_ptr<Engine<A>> e;
    TRY(Engine<A>::open(std::move(t), false, e));
    pn_build_opts o{};
    o.algo = e->tree->algo;
    return finish_create<A>(kind, e, o, t0, out);
}

template <typename A>
static int merge_topk_dev(int device, const uint64_t* idx_lists, const A* dist_lists, size_t n_lists, size_t nq, size_t k,
                          uint64_t* idx_out, A* dist_out, cudaStream_t st, bool sync) {
    if (!idx_lists || !dist_lists || !idx_out || !dist_out) return fail(PN_BAD_ARG, "null pointer");
    if (n_lists == 0 || n_lists > (size_t)MAX_LISTS) return fail(PN_BAD_ARG, "n_lists must be in 1..256");
    if (k > 65535 || nq >= (1ull << 32)) return fail(PN_BAD_ARG, "k must be <= 65535 and nq < 2^32");
    if (nq == 0 || k == 0) return PN_OK;
    DeviceGuard g(device);
    if (!g.ok) return fail(PN_CUDA, "cudaSetDevice failed");
    CU(merge_lists<A, uint64_t>(st, dist_lists, idx_lists, (uint32_t)n_lists, (uint32_t)nq,
                                                                          (uint32_t)k, idx_out, dist_out, (uint32_t)k, 0, nullptr, nullptr));
    CU(cudaGetLastError());
    if (sync) CU(cudaStreamSynchronize(st));
    return PN_OK;
}

static int merge_radius_dev(int device, const uint64_t* offsets, const uint64_t* indices, size_t n_lists, size_t nq, uint64_t* out_offsets,
                            uint64_t* out_indices, cudaStream_t st, bool sync) {
    if (!offsets || !indices || !out_offsets || !out_indices) return fail(PN_BAD_ARG, "null pointer");
    if (n_lists == 0 || n_lists > (size_t)MAX_LISTS) return fail(PN_BAD_ARG, "n_lists must be in 1..256");
    if (nq >= (1ull << 32)) return fail(PN_BAD_ARG, "nq must be < 2^32");
    DeviceGuard g(device);
    if (!g.ok) return fail(PN_CUDA, "cudaSetDevice failed");
    if (nq == 0) {
        CU(cudaMemsetAsync(out_offsets, 0, 8, st));
    } else {
        int n_sms = 0;
        CU(cudaDeviceGetAttribute(&n_sms, cudaDevAttrMultiProcessorCount, device));
        // stream-ordered workspace (sums, then the u32 counts), so the call does not synchronise the device
        const size_t sums_bytes = ((nq / SCAN_BLOCK + 1) * 8 + 255) / 256 * 256;
        void* ws = nullptr;
        CU(cudaMallocAsync(&ws, sums_bytes + nq * 4, st));
        const cudaError_t e = merge_radius_lists<uint64_t>(st, offsets, indices, (uint32_t)n_lists, (uint32_t)nq, out_offsets, out_indices,
                                                           (uint32_t*)((char*)ws + sums_bytes), (unsigned long long*)ws, 8u * (unsigned)n_sms);
        const cudaError_t ef = cudaFreeAsync(ws, st);
        CU(e);
        CU(ef);
    }
    if (sync) CU(cudaStreamSynchronize(st));
    return PN_OK;
}

template <typename A>
static int pairwise_host(int device, const A* x, size_t n, size_t d, size_t row_stride, A* out) {
    if (n == 0) return PN_OK;
    if (!x || !out) return fail(PN_BAD_ARG, "null pointer");
    if (d == 0 || n >= (1ull << 31) || (n > 1 && row_stride < d)) return fail(PN_BAD_ARG, "bad shape");
    int dev = device;
    if (dev < 0 && cudaGetDevice(&dev) != cudaSuccess) { (void)cudaGetLastError(); return fail(PN_CUDA, "no CUDA device available (there is no CPU fallback)"); }
    DeviceGuard g(dev);
    if (!g.ok) return fail(PN_CUDA, "cudaSetDevice failed");
    // the matrix leaves the device in row blocks of at most 256 MiB, so n is bounded by the caller's host buffer, not by HBM
    DevBuf dx, dout;
    const size_t rows_per_block = std::max<size_t>(32, std::min<size_t>(n, ((size_t)256 << 20) / (n * sizeof(A)) / 32 * 32));
    int rc = dx.ensure(n * d * sizeof(A));
    if (rc == PN_OK) rc = dout.ensure(rows_per_block * n * sizeof(A));
    if (rc == PN_OK) {
        cudaError_t e = cudaMemcpy2D(dx.p, d * sizeof(A), x, row_stride * sizeof(A), d * sizeof(A), n, cudaMemcpyHostToDevice);
        for (size_t r0 = 0; r0 < n && e == cudaSuccess; r0 += rows_per_block) {
            const size_t rows = std::min(rows_per_block, n - r0);
            dim3 grid((unsigned)((n + 31) / 32), (unsigned)((rows + 31) / 32)), block(32, 32);
            pairwise_kernel<A><<<grid, block>>>(dx.as<A>(), (uint32_t)n, (uint32_t)d, dout.as<A>(), (uint32_t)r0, (uint32_t)rows);
            e = cudaGetLastError();
            if (e == cudaSuccess) e = cudaMemcpy(out + r0 * n, dout.p, rows * n * sizeof(A), cudaMemcpyDeviceToHost);
        }
        if (e != cudaSuccess) rc = fail(PN_CUDA, std::string("pairwise: ") + cudaGetErrorString(e));
    }
    return rc;
}

}  // namespace petal

// ================================= C ABI ======================================================
#define GUARD_BEGIN try {
#define GUARD_END                                                              \
    }                                                                          \
    catch (const std::bad_alloc&) { return fail(PN_OOM, "host allocation failed"); } \
    catch (const std::exception& ex) { return fail(PN_BAD_ARG, ex.what()); }  \
    catch (...) { return fail(PN_BAD_ARG, "unknown error"); }

static int check_tree(const pn_tree* t, uint32_t dtype, int kind) {
    if (!t) return fail(PN_BAD_ARG, "tree is null");
    if (t->info.dtype != dtype) return fail(PN_BAD_ARG, "element type of the call does not match the tree");
    if (kind >= 0 && (int)t->info.kind != kind) return fail(PN_BAD_ARG, "tree kind does not match the call");
    return PN_OK;
}

extern "C" {

const char* pn_last_error_message(void) { return g_err.c_str(); }
int32_t pn_abi_version(void) { return PN_ABI_VERSION; }
int32_t pn_device_count(int32_t* count) {
    if (!count) return fail(PN_BAD_ARG, "count is null");
    int c = 0;
    if (cudaGetDeviceCount(&c) != cudaSuccess) { (void)cudaGetLastError(); c = 0; }
    *count = c;
    return PN_OK;
}

int32_t pn_balltree_create_f32(const float* p, size_t n, size_t d, size_t rs, size_t cs, const pn_build_opts* o, pn_tree** out) {
    GUARD_BEGIN return create_tree<float>(PN_KIND_BALL, p, n, d, rs, cs, o, out); GUARD_END
}
int32_t pn_balltree_create_f64(const double* p, size_t n, size_t d, size_t rs, size_t cs, const pn_build_opts* o, pn_tree** out) {
    GUARD_BEGIN return create_tree<double>(PN_KIND_BALL, p, n, d, rs, cs, o, out); GUARD_END
}
int32_t pn_vptree_create_f32(const float* p, size_t n, size_t d, size_t rs, size_t cs, const pn_build_opts* o, pn_tree** out) {
    GUARD_BEGIN return create_tree<float>(PN_KIND_VP, p, n, d, rs, cs, o, out); GUARD_END
}
int32_t pn_vptree_create_f64(const double* p, size_t n, size_t d, size_t rs, size_t cs, const pn_build_opts* o, pn_tree** out) {
    GUARD_BEGIN return create_tree<double>(PN_KIND_VP, p, n, d, rs, cs, o, out); GUARD_END
}
int32_t pn_balltree_create_dev_f32(const float* p, size_t n, size_t d, size_t rs, const pn_build_opts* o, pn_tree** out) {
    GUARD_BEGIN return create_tree_dev<float>(p, n, d, rs, o, out); GUARD_END
}
int32_t pn_balltree_create_dev_f64(const double* p, size_t n, size_t d, size_t rs, const pn_build_opts* o, pn_tree** out) {
    GUARD_BEGIN return create_tree_dev<double>(p, n, d, rs, o, out); GUARD_END
}
int32_t pn_tree_destroy(pn_tree* t) {
    GUARD_BEGIN
    delete t;   // the tree itself is freed with the last handle that shares it
    return PN_OK;
    GUARD_END
}
int32_t pn_tree_session(pn_tree* t, pn_tree** out) {
    GUARD_BEGIN
    if (!t || !out) return fail(PN_BAD_ARG, "null argument");
    *out = nullptr;
    return t->session(out);
    GUARD_END
}

int32_t pn_balltree_query_f32(pn_tree* t, const float* q, size_t nq, size_t qs, size_t k, uint64_t* io, float* dd) {
    GUARD_BEGIN TRY(check_tree(t, PN_F32, PN_KIND_BALL)); return t->knn_host(q, nq, qs, k, io, dd); GUARD_END
}
int32_t pn_balltree_query_f64(pn_tree* t, const double* q, size_t nq, size_t qs, size_t k, uint64_t* io, double* dd) {
    GUARD_BEGIN TRY(check_tree(t, PN_F64, PN_KIND_BALL)); return t->knn_host(q, nq, qs, k, io, dd); GUARD_END
}
int32_t pn_balltree_query_nearest_f32(pn_tree* t, const float* q, size_t nq, size_t qs, uint64_t* io, float* dd) {
    GUARD_BEGIN TRY(check_tree(t, PN_F32, PN_KIND_BALL)); return t->knn_host(q, nq, qs, 1, io, dd); GUARD_END
}
int32_t pn_balltree_query_nearest_f64(pn_tree* t, const double* q, size_t nq, size_t qs, uint64_t* io, double* dd) {
    GUARD_BEGIN TRY(check_tree(t, PN_F64, PN_KIND_BALL)); return t->knn_host(q, nq, qs, 1, io, dd); GUARD_END
}
int32_t pn_balltree_query_radius_f32(pn_tree* t, const float* q, size_t nq, size_t qs, float r, uint64_t** oo, uint64_t** io) {
    GUARD_BEGIN TRY(check_tree(t, PN_F32, PN_KIND_BALL)); return t->radius_host(q, nq, qs, (double)r, oo, io); GUARD_END
}
int32_t pn_balltree_query_radius_f64(pn_tree* t, const double* q, size_t nq, size_t qs, double r, uint64_t** oo, uint64_t** io) {
    GUARD_BEGIN TRY(check_tree(t, PN_F64, PN_KIND_BALL)); return t->radius_host(q, nq, qs, r, oo, io); GUARD_END
}
int32_t pn_vptree_query_nearest_f32(pn_tree* t, const float* q, size_t nq, size_t qs, uint64_t* io, float* dd) {
    GUARD_BEGIN TRY(check_tree(t, PN_F32, PN_KIND_VP)); return t->knn_host(q, nq, qs, 1, io, dd); GUARD_END
}
int32_t pn_vptree_query_nearest_f64(pn_tree* t, const double* q, size_t nq, size_t qs, uint64_t* io, double* dd) {
    GUARD_BEGIN TRY(check_tree(t, PN_F64, PN_KIND_VP)); return t->knn_host(q, nq, qs, 1, io, dd); GUARD_END
}
int32_t pn_vptree_query_f32(pn_tree* t, const float* q, size_t nq, size_t qs, size_t k, uint64_t* io, float* dd) {
    GUARD_BEGIN TRY(check_tree(t, PN_F32, PN_KIND_VP)); return t->knn_host(q, nq, qs, k, io, dd); GUARD_END
}
int32_t pn_vptree_query_f64(pn_tree* t, const double* q, size_t nq, size_t qs, size_t k, uint64_t* io, double* dd) {
    GUARD_BEGIN TRY(check_tree(t, PN_F64, PN_KIND_VP)); return t->knn_host(q, nq, qs, k, io, dd); GUARD_END
}
int32_t pn_vptree_query_radius_f32(pn_tree* t, const float* q, size_t nq, size_t qs, float r, uint64_t** oo, uint64_t** io) {
    GUARD_BEGIN TRY(check_tree(t, PN_F32, PN_KIND_VP)); return t->radius_host(q, nq, qs, (double)r, oo, io); GUARD_END
}
int32_t pn_vptree_query_radius_f64(pn_tree* t, const double* q, size_t nq, size_t qs, double r, uint64_t** oo, uint64_t** io) {
    GUARD_BEGIN TRY(check_tree(t, PN_F64, PN_KIND_VP)); return t->radius_host(q, nq, qs, r, oo, io); GUARD_END
}
int32_t pn_balltree_query_self_f32(pn_tree* t, size_t k, uint64_t* io, float* dd) {
    GUARD_BEGIN TRY(check_tree(t, PN_F32, PN_KIND_BALL)); return t->knn_self(k, io, dd, false, nullptr, true); GUARD_END
}
int32_t pn_balltree_query_self_f64(pn_tree* t, size_t k, uint64_t* io, double* dd) {
    GUARD_BEGIN TRY(check_tree(t, PN_F64, PN_KIND_BALL)); return t->knn_self(k, io, dd, false, nullptr, true); GUARD_END
}
int32_t pn_tree_query_self_dev(pn_tree* t, size_t k, uint64_t* io, void* dd, void* stream, int32_t sync) {
    GUARD_BEGIN
    if (!t) return fail(PN_BAD_ARG, "tree is null");
    return t->knn_self(k, io, dd, true, (cudaStream_t)stream, sync != 0);
    GUARD_END
}
int32_t pn_pairwise_f32(int32_t device, const float* x, size_t n, size_t d, size_t row_stride, float* out) {
    GUARD_BEGIN return pairwise_host<float>(device, x, n, d, row_stride, out); GUARD_END
}
int32_t pn_pairwise_f64(int32_t device, const double* x, size_t n, size_t d, size_t row_stride, double* out) {
    GUARD_BEGIN return pairwise_host<double>(device, x, n, d, row_stride, out); GUARD_END
}
void pn_free(void* p) { free(p); }

int32_t pn_tree_query_knn_dev(pn_tree* t, const void* q, size_t nq, size_t qs, size_t k, uint64_t* io, void* dd, void* stream, int32_t sync) {
    GUARD_BEGIN
    if (!t) return fail(PN_BAD_ARG, "tree is null");
    return t->knn_dev(q, nq, qs, k, io, dd, (cudaStream_t)stream, sync != 0);
    GUARD_END
}
int32_t pn_tree_query_radius_dev(pn_tree* t, const void* q, size_t nq, size_t qs, double radius, uint64_t* oo, uint64_t* io, size_t capacity,
                                 void* stream, int32_t sync) {
    GUARD_BEGIN
    if (!t) return fail(PN_BAD_ARG, "tree is null");
    return t->radius_dev(q, nq, qs, radius, oo, io, capacity, (cudaStream_t)stream, sync != 0);
    GUARD_END
}
int32_t pn_merge_topk_dev(uint32_t dtype, int32_t device, const uint64_t* il, const void* dl, size_t n_lists, size_t nq, size_t k,
                          uint64_t* io, void* dd, void* stream, int32_t sync) {
    GUARD_BEGIN
    if (dtype == PN_F32) return merge_topk_dev<float>(device, il, (const float*)dl, n_lists, nq, k, io, (float*)dd, (cudaStream_t)stream, sync != 0);
    if (dtype == PN_F64) return merge_topk_dev<double>(device, il, (const double*)dl, n_lists, nq, k, io, (double*)dd, (cudaStream_t)stream, sync != 0);
    return fail(PN_BAD_ARG, "bad dtype");
    GUARD_END
}

int32_t pn_merge_radius_dev(int32_t device, const uint64_t* ol, const uint64_t* il, size_t n_lists, size_t nq, uint64_t* oo, uint64_t* io,
                            void* stream, int32_t sync) {
    GUARD_BEGIN return merge_radius_dev(device, ol, il, n_lists, nq, oo, io, (cudaStream_t)stream, sync != 0); GUARD_END
}

// ---- multi-GPU: communicator ranks, sharded k-NN, replication ---------------------------------------------------------
void pn_query_slice(size_t nq, int32_t rank, int32_t world, size_t* lo, size_t* hi) {
    if (world < 1) world = 1;
    const size_t base = nq / (size_t)world, rem = nq % (size_t)world, r = (size_t)std::max(rank, 0);
    const size_t l = r * base + std::min(r, rem);
    if (lo) *lo = l;
    if (hi) *hi = l + base + (r < rem ? 1 : 0);
}
int32_t pn_comm_unique_id(void* id_out) {
    GUARD_BEGIN
    if (!id_out) return fail(PN_BAD_ARG, "id_out is null");
    std::string err;
    NcclApi* api = NcclApi::get(&err);
    if (!api) return fail(PN_NCCL, err);
    static_assert(sizeof(ncclUniqueId) == PN_UNIQUE_ID_BYTES, "unique id size");
    ncclUniqueId id;
    ncclResult_t r = api->GetUniqueId(&id);
    if (r != ncclSuccess) return fail(PN_NCCL, std::string("ncclGetUniqueId: ") + api->GetErrorString(r));
    memcpy(id_out, &id, sizeof(id));
    return PN_OK;
    GUARD_END
}
static int finish_comm(pn_comm* c) {
    DeviceGuard g(c->device);
    if (!g.ok) return fail(PN_CUDA, "cudaSetDevice failed");
    CU(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    return PN_OK;
}
int32_t pn_comm_create(const void* unique_id, int32_t world, int32_t rank, int32_t device, pn_comm** out) {
    GUARD_BEGIN
    if (!out) return fail(PN_BAD_ARG, "out is null");
    *out = nullptr;
    if (!unique_id || world < 1 || rank < 0 || rank >= world) return fail(PN_BAD_ARG, "bad unique id / world / rank");
    std::string err;
    NcclApi* api = NcclApi::get(&err);
    if (!api) return fail(PN_NCCL, err);
    if (device < 0 && cudaGetDevice(&device) != cudaSuccess) { (void)cudaGetLastError(); return fail(PN_CUDA, "no CUDA device available"); }
    std::unique_ptr<pn_comm> c(new pn_comm());
    c->api = api; c->world = world; c->rank = rank; c->device = device;
    {
        DeviceGuard g(device);
        if (!g.ok) return fail(PN_CUDA, "cudaSetDevice failed");
        ncclUniqueId id;
        memcpy(&id, unique_id, sizeof(id));
        ncclResult_t r = api->CommInitRank(&c->comm, world, id, rank);
        if (r != ncclSuccess) return fail(PN_NCCL, std::string("ncclCommInitRank: ") + api->GetErrorString(r));
    }
    TRY(finish_comm(c.get()));
    *out = c.release();
    return PN_OK;
    GUARD_END
}
int32_t pn_comm_create_all(const int32_t* devices, int32_t n_dev, pn_comm** out) {
    GUARD_BEGIN
    if (!out || !devices || n_dev < 1 || n_dev > 64) return fail(PN_BAD_ARG, "bad device list");
    std::string err;
    NcclApi* api = NcclApi::get(&err);
    if (!api) return fail(PN_NCCL, err);
    std::vector<ncclComm_t> comms(n_dev);
    std::vector<int> devs(devices, devices + n_dev);
    ncclResult_t r = api->CommInitAll(comms.data(), n_dev, devs.data());
    if (r != ncclSuccess) return fail(PN_NCCL, std::string("ncclCommInitAll: ") + api->GetErrorString(r));
    for (int i = 0; i < n_dev; ++i) {
        pn_comm* c = new pn_comm();
        c->api = api; c->comm = comms[i]; c->world = n_dev; c->rank = i; c->device = devs[i];
        out[i] = c;
        TRY(finish_comm(c));
    }
    return PN_OK;
    GUARD_END
}
int32_t pn_comm_destroy(pn_comm* c) {
    GUARD_BEGIN
    if (!c) return PN_OK;
    DeviceGuard g(c->device);
    if (c->stream) { cudaStreamSynchronize(c->stream); cudaStreamDestroy(c->stream); }
    if (c->comm) c->api->CommDestroy(c->comm);
    delete c;
    return PN_OK;
    GUARD_END
}
int32_t pn_sharded_query_knn_dev(pn_tree* t, pn_comm* comm, const void* q, size_t nq, size_t qs, size_t k, uint32_t exchange, uint64_t* io,
                                 void* dd, void* stream, pn_shard_stats* stats) {
    GUARD_BEGIN
    if (!t) return fail(PN_BAD_ARG, "tree is null");
    if (t->info.kind != PN_KIND_BALL) return fail(PN_BAD_ARG, "point sharding by subtree is a ball-tree feature");
    return t->knn_sharded(comm, q, nq, qs, k, exchange, io, dd, (cudaStream_t)stream, stats);
    GUARD_END
}
int32_t pn_tree_replicate(pn_tree* t, pn_comm* cm, int32_t root, pn_tree** out) {
    GUARD_BEGIN
    if (!cm || !out) return fail(PN_BAD_ARG, "null pointer");
    if (root < 0 || root >= cm->world) return fail(PN_BAD_ARG, "bad root");
    *out = nullptr;
    const bool is_root = cm->rank == root;
    if (is_root && !t) return fail(PN_BAD_ARG, "the root rank needs a tree");
    DeviceGuard g(cm->device);
    if (!g.ok) return fail(PN_CUDA, "cudaSetDevice failed");
    // element type and kind first: the receivers need them to make their handle
    int32_t meta[2] = {is_root ? (int32_t)t->info.dtype : 0, is_root ? (int32_t)t->info.kind : 0};
    DevBuf mb;
    TRY(mb.ensure(sizeof(meta)));
    CU(cudaMemcpyAsync(mb.p, meta, sizeof(meta), cudaMemcpyHostToDevice, cm->stream));
    ncclResult_t r = cm->api->Broadcast(mb.p, mb.p, sizeof(meta), ncclUint8, root, cm->comm, cm->stream);
    if (r != ncclSuccess) return fail(PN_NCCL, std::string("ncclBroadcast: ") + cm->api->GetErrorString(r));
    CU(cudaMemcpyAsync(meta, mb.p, sizeof(meta), cudaMemcpyDeviceToHost, cm->stream));
    CU(cudaStreamSynchronize(cm->stream));
    if (is_root) {
        TRY(t->replicate_send(cm, root));
        *out = t;
        return PN_OK;
    }
    return meta[0] == PN_F32 ? receive_replica<float>(cm, root, meta[1], out) : receive_replica<double>(cm, root, meta[1], out);
    GUARD_END
}

// ---- one process, several GPUs ---------------------------------------------------------------------------------------
}  // extern "C"
struct pn_multi {
    int n_dev = 0;
    uint32_t mode = PN_SHARD_REPLICATE;
    size_t d = 0;
    std::vector<int> devices;
    std::vector<pn_comm*> comms;
    std::vector<pn_tree*> trees;
    std::vector<pn_shard_stats> stats;
    std::vector<DevBuf> q_dev, idx_dev, dist_dev;  // BY_SUBTREE: all queries / this device's result slice
    PeerShared peer;                                // PEER exchange: shared by the rank threads of a query
    bool peer_ok = false;                           // every pair of devices has peer access
    uint32_t exchange = PN_EXCHANGE_SLICE;
    ~pn_multi() {
        for (size_t i = 0; i < trees.size(); ++i) {
            if (!trees[i]) continue;
            bool dup = false;
            for (size_t j = 0; j < i; ++j) dup |= trees[j] == trees[i];
            if (!dup) delete trees[i];
        }
        for (pn_comm* c : comms) pn_comm_destroy(c);
    }
};
// fn(rank) on one host thread per rank; the first failure (status + message) is reported in the caller's thread
template <typename F>
static int on_every_rank(int n, F fn) {
    std::vector<int> rc(n, PN_OK);
    std::vector<std::string> msg(n);
    std::vector<std::thread> th;
    for (int r = 0; r < n; ++r)
        th.emplace_back([&, r] {
            try { rc[r] = fn(r); } catch (const std::exception& ex) { rc[r] = fail(PN_BAD_ARG, ex.what()); } catch (...) { rc[r] = fail(PN_BAD_ARG, "unknown error"); }
            if (rc[r] != PN_OK) msg[r] = g_err;
        });
    for (auto& t : th) t.join();
    int first = -1;   // the first rank that failed on its own, else the first that was released by another's failure
    for (int r = n - 1; r >= 0; --r)
        if (rc[r] != PN_OK && (first < 0 || msg[r] != PeerShared::RELEASED || msg[first] == PeerShared::RELEASED)) first = r;
    if (first >= 0) return fail(rc[first], "device rank " + std::to_string(first) + ": " + msg[first]);
    return PN_OK;
}
extern "C" {
int32_t pn_multi_balltree_create_f32(const int32_t* devices, int32_t n_dev, uint32_t mode, const float* points, size_t n, size_t d, size_t rs,
                                     const pn_build_opts* opts_in, pn_multi** out) {
    GUARD_BEGIN
    if (!out) return fail(PN_BAD_ARG, "out is null");
    *out = nullptr;
    if (!devices || n_dev < 1 || n_dev > 64) return fail(PN_BAD_ARG, "bad device list");
    if (mode > PN_SHARD_BY_SUBTREE) return fail(PN_BAD_ARG, "bad shard mode");
    uint32_t depth = 0;
    while ((1 << depth) < n_dev) ++depth;
    if (mode == PN_SHARD_BY_SUBTREE && (1 << depth) != n_dev) return fail(PN_BAD_ARG, "sharding by subtree needs a power-of-two number of devices");
    pn_build_opts o = read_build_opts(opts_in);
    o.struct_size = sizeof(o);
    if (o.flags & PN_FLAG_HOST_ONLY) return fail(PN_BAD_ARG, "a multi-GPU tree cannot be host-only");
    std::unique_ptr<pn_multi> m(new pn_multi());
    m->n_dev = n_dev; m->mode = mode; m->d = d;
    m->devices.assign(devices, devices + n_dev);
    m->comms.assign(n_dev, nullptr);
    m->trees.assign(n_dev, nullptr);
    m->stats.assign(n_dev, pn_shard_stats{});
    m->q_dev.resize(n_dev); m->idx_dev.resize(n_dev); m->dist_dev.resize(n_dev);
    m->peer.n = n_dev;
    TRY(pn_comm_create_all(devices, n_dev, m->comms.data()));
    if (mode == PN_SHARD_REPLICATE) {
        pn_build_opts o0 = o;
        o0.device = devices[0]; o0.shard_depth = 0; o0.shard_index = 0;
        TRY(pn_balltree_create_f32(points, n, d, rs, 1, &o0, &m->trees[0]));
        TRY(on_every_rank(n_dev, [&](int r) { return (int)pn_tree_replicate(r == 0 ? m->trees[0] : nullptr, m->comms[r], 0, &m->trees[r]); }));
    } else {
        TRY(on_every_rank(n_dev, [&](int r) {
            pn_build_opts orr = o;
            orr.device = devices[r]; orr.shard_depth = depth; orr.shard_index = (uint32_t)r;
            return (int)pn_balltree_create_f32(points, n, d, rs, 1, &orr, &m->trees[r]);
        }));
        // peer access between every pair of devices: the merge kernels then read the other shards' lists in place
        m->peer_ok = true;
        for (int i = 0; i < n_dev; ++i)
            for (int j = 0; j < n_dev; ++j) {
                if (devices[i] == devices[j]) continue;
                int can = 0;
                if (cudaDeviceCanAccessPeer(&can, devices[i], devices[j]) != cudaSuccess || !can) { m->peer_ok = false; continue; }
                DeviceGuard g(devices[i]);
                cudaError_t e = cudaDeviceEnablePeerAccess(devices[j], 0);
                if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) m->peer_ok = false;
                (void)cudaGetLastError();
            }
        m->peer.pack.assign(n_dev, nullptr);
        m->peer.ev_scan.resize(n_dev);
        if (m->peer_ok) m->exchange = PN_EXCHANGE_PEER;
    }
    *out = m.release();
    return PN_OK;
    GUARD_END
}
int32_t pn_multi_balltree_query_f32(pn_multi* m, const float* q, size_t nq, size_t qs, size_t k, uint64_t* idx_out, float* dist_out) {
    GUARD_BEGIN
    if (!m) return fail(PN_BAD_ARG, "handle is null");
    if (nq == 0 || k == 0) return PN_OK;
    if (!q || !idx_out || !dist_out) return fail(PN_BAD_ARG, "null pointer");
    if (nq > 1 && qs < m->d) return fail(PN_BAD_ARG, "q_row_stride < dimension");
    const int W = m->n_dev;
    { std::lock_guard<std::mutex> lk(m->peer.mu); m->peer.failed = false; m->peer.count = 0; }
    if (m->mode == PN_SHARD_BY_SUBTREE && m->exchange == PN_EXCHANGE_PEER) {
        // the chunking of this call and one scan event per (rank, chunk), created on the rank's device
        m->peer.chunk = m->trees[0]->shard_chunk(nq);
        m->peer.n_chunks = (nq + m->peer.chunk - 1) / m->peer.chunk;
        for (int r = 0; r < W; ++r) {
            DeviceGuard g(m->devices[r]);
            TRY(grow_events(m->peer.ev_scan[r], m->peer.n_chunks, cudaEventDisableTiming));
        }
    }
    return on_every_rank(W, [&](int r) -> int {
        size_t lo, hi;
        pn_query_slice(nq, r, W, &lo, &hi);
        m->stats[r] = pn_shard_stats{};
        m->stats[r].rows_out = hi - lo;
        if (m->mode == PN_SHARD_REPLICATE) {
            if (hi == lo) return PN_OK;
            return pn_balltree_query_f32(m->trees[r], q + lo * qs, hi - lo, qs, k, idx_out + lo * k, dist_out + lo * k);
        }
        // BY_SUBTREE: all queries on every device, the merged rows of this device's slice come back
        DeviceGuard g(m->devices[r]);
        if (!g.ok) return fail(PN_CUDA, "cudaSetDevice failed");
        const size_t d = m->d, rows = hi - lo;
        TRY(m->q_dev[r].ensure(nq * d * 4));
        TRY(m->idx_dev[r].ensure(std::max<size_t>(rows, 1) * k * 8));
        TRY(m->dist_dev[r].ensure(std::max<size_t>(rows, 1) * k * 4));
        CU(cudaMemcpy2D(m->q_dev[r].p, d * 4, q, std::max(qs, d) * 4, d * 4, nq, cudaMemcpyHostToDevice));
        if (m->exchange == PN_EXCHANGE_PEER) {
            TRY(m->trees[r]->knn_sharded_peer(m->peer, r, W, m->q_dev[r].p, nq, d, k, m->idx_dev[r].as<uint64_t>(), m->dist_dev[r].p, &m->stats[r]));
        } else {
            TRY(pn_sharded_query_knn_dev(m->trees[r], m->comms[r], m->q_dev[r].p, nq, d, k, PN_EXCHANGE_SLICE, m->idx_dev[r].as<uint64_t>(),
                                         m->dist_dev[r].p, nullptr, &m->stats[r]));
        }
        if (rows) {
            CU(cudaMemcpy(idx_out + lo * k, m->idx_dev[r].p, rows * k * 8, cudaMemcpyDeviceToHost));
            CU(cudaMemcpy(dist_out + lo * k, m->dist_dev[r].p, rows * k * 4, cudaMemcpyDeviceToHost));
        }
        return PN_OK;
    });
    GUARD_END
}
int32_t pn_multi_balltree_query_radius_f32(pn_multi* m, const float* q, size_t nq, size_t qs, float radius, uint64_t** offsets_out,
                                           uint64_t** indices_out) {
    GUARD_BEGIN
    if (!offsets_out || !indices_out) return fail(PN_BAD_ARG, "output pointer is null");
    if (nq && !q) return fail(PN_BAD_ARG, "queries is null");
    if (nq >= (1ull << 32)) return fail(PN_BAD_ARG, "nq must be < 2^32 per call");
    if (!m) return fail(PN_BAD_ARG, "handle is null");
    if (nq > 1 && qs < m->d) return fail(PN_BAD_ARG, "q_row_stride < dimension");
    const int W = m->n_dev;
    for (int r = 0; r < W; ++r) m->stats[r] = pn_shard_stats{};
    PeerShared& ps = m->peer;
    { std::lock_guard<std::mutex> lk(ps.mu); ps.failed = false; ps.count = 0; }
    ps.r_offs.assign(W, nullptr); ps.r_hits.assign(W, nullptr); ps.r_dev.assign(W, -1);
    ps.r_bound.assign(W, {}); ps.r_total.assign(W, 0);
    ps.r_out_offs = nullptr; ps.r_out_hits = nullptr;
    int rc = PN_OK;
    if (nq == 0) {   // as pn_balltree_query_radius_f32: offsets {0} and an empty index array, both for pn_free
        ps.r_out_offs = (uint64_t*)malloc(8);
        ps.r_out_hits = (uint64_t*)malloc(8);
        if (ps.r_out_offs) ps.r_out_offs[0] = 0;
        if (!ps.r_out_offs || !ps.r_out_hits) rc = fail(PN_OOM, "malloc offsets");
    } else {
        rc = on_every_rank(W, [&](int r) -> int {
            return m->trees[r]->radius_multi(ps, r, W, m->mode == PN_SHARD_BY_SUBTREE, q, nq, qs, (double)radius, &m->stats[r]);
        });
    }
    if (rc != PN_OK) {
        free(ps.r_out_offs); free(ps.r_out_hits);
        ps.r_out_offs = nullptr; ps.r_out_hits = nullptr;
        return rc;
    }
    *offsets_out = ps.r_out_offs; *indices_out = ps.r_out_hits;
    ps.r_out_offs = nullptr; ps.r_out_hits = nullptr;
    return PN_OK;
    GUARD_END
}
int32_t pn_multi_set_exchange(pn_multi* m, uint32_t exchange) {
    if (!m) return fail(PN_BAD_ARG, "handle is null");
    if (exchange != PN_EXCHANGE_SLICE && exchange != PN_EXCHANGE_PEER) return fail(PN_BAD_ARG, "the exchange of a multi-GPU handle is SLICE or PEER");
    if (exchange == PN_EXCHANGE_PEER && !m->peer_ok) return fail(PN_BAD_ARG, "peer access is not available between every pair of devices");
    m->exchange = exchange;
    return PN_OK;
}
int32_t pn_multi_get_stats(const pn_multi* m, pn_shard_stats* stats, int32_t n_stats) {
    if (!m || !stats) return fail(PN_BAD_ARG, "null pointer");
    for (int r = 0; r < std::min<int>(n_stats, m->n_dev); ++r) stats[r] = m->stats[r];
    return PN_OK;
}
int32_t pn_multi_destroy(pn_multi* m) {
    GUARD_BEGIN delete m; return PN_OK; GUARD_END
}

int32_t pn_tree_get_info(const pn_tree* t, pn_tree_info* info) {
    if (!t || !info) return fail(PN_BAD_ARG, "null pointer");
    *info = t->info;
    info->device_bytes = t->device_bytes();
    return PN_OK;
}
int32_t pn_tree_get_counters(const pn_tree* t, pn_counters* c) {
    if (!t || !c) return fail(PN_BAD_ARG, "null pointer");
    *c = t->counters;
    return PN_OK;
}
int32_t pn_tree_get_layout(const pn_tree* t, uint32_t* ids, uint32_t* blo, uint32_t* bhi, void* rad, void* cen, void* pts) {
    GUARD_BEGIN
    if (!t) return fail(PN_BAD_ARG, "tree is null");
    return const_cast<pn_tree*>(t)->layout(ids, blo, bhi, rad, cen, pts);
    GUARD_END
}

}  // extern "C"
