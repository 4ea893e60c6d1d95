// gpu_build.hpp -- device-side construction of the flattened ball tree (SURVEY.md 8f row 2).
//
// The same partition as the host builder of flat_tree.hpp (reference: build_subtree src/ball_tree.rs:504-538,
// Node::init :445-461, max_spread_column :577-613, halve_node_indices :545-569), produced level by level on the GPU:
//   per level : segmented per-column min/max -> max-spread column (first strictly greatest wins) -> the median of the
//               segment by a radix select on the (value, index) key -> stable partition around it
//   then      : gather of the rows in bucket order, bucket sums -> centroids bottom-up, radii in one pass over the rows.
// Within a bucket the points are stored in ascending original index on both builders, so the two layouts are
// bit-identical (tests/test_gpu_build.py) -- exact query results never depended on the layout anyway.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <mutex>
#include <set>
#include <string>
#include <utility>
#include <vector>

namespace petal {

// Lets `kern` launch with as much dynamic shared memory as the current device offers a block.  The limit a launch is
// checked against is state of the kernel shared by every thread of the process: if each caller set the size it needs,
// a caller on another thread (another session, another tree) could lower it between this caller's setting and its
// launch, which then fails with cudaErrorInvalidValue.  Every caller sets the same value instead, once per kernel and
// device: later calls cost a cudaGetDevice and a lookup.
template <typename F>
inline cudaError_t allow_max_dynamic_smem(F* kern) {
    static std::mutex mu;
    static std::set<std::pair<const void*, int>> done;   // (kernel, device) pairs whose limit is raised
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    const std::pair<const void*, int> key((const void*)kern, dev);
    std::lock_guard<std::mutex> lk(mu);
    if (done.count(key)) return cudaSuccess;
    int optin = 0;
    cudaFuncAttributes fa{};
    e = cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    if (e == cudaSuccess) e = cudaFuncGetAttributes(&fa, kern);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, optin - (int)fa.sharedSizeBytes);
    if (e == cudaSuccess) done.insert(key);
    return e;
}

namespace gb {

// Shape of the implicit complete tree over n points cut at level L (host arithmetic only, shared by both builders):
// seg[l] holds the 2^l + 1 boundaries of the level-l nodes in the bucket-ordered point array, by the reference's
// mid = (start + end) / 2 rule (src/ball_tree.rs:535-537).
struct TreeShape {
    uint64_t n = 0;
    uint32_t L = 0;
    std::vector<std::vector<uint32_t>> seg;  // [L + 1][2^l + 1]
    uint32_t align = 0;  // > 0 (two-means partition only): nodes of more than one `align`-row tile split between tiles,
                         // floor(tiles / 2) of them to the left, so every node starts on a multiple of `align`
    void init(uint64_t n_, uint32_t L_, uint32_t align_ = 0) {
        n = n_; L = L_; align = align_;
        seg.assign(L + 1, {});
        seg[0] = {0u, (uint32_t)n};
        for (uint32_t l = 0; l < L; ++l) {
            const auto& a = seg[l];
            auto& b = seg[l + 1];
            b.resize((size_t(1) << (l + 1)) + 1);
            for (size_t s = 0; s + 1 < a.size(); ++s) {
                b[2 * s] = a[s];
                b[2 * s + 1] = (uint32_t)(((uint64_t)a[s] + a[s + 1]) / 2);
                if (align) {
                    const uint32_t tiles = (a[s + 1] - a[s] + align - 1) / align;
                    if (tiles >= 2) b[2 * s + 1] = a[s] + align * (tiles / 2);
                }
            }
            b[size_t(1) << (l + 1)] = (uint32_t)n;
        }
    }
};

// Device arrays the builder fills (all allocated by the caller):
template <typename A>
struct BallOut {
    A* pts;          // n x dpad, bucket order, zero padded
    uint32_t* ids;   // n
    A* centers;      // n_nodes x dpad
    A* radii;        // n_nodes (-1 = empty node)
    A* plane_w = nullptr;  // two-means rule only (optional): n_internal x dpad split directions ...
    A* plane_t = nullptr;  // ... and n_internal pivot keys: a row with  row . w < t  went to the left child
};

// raw: n_all x d rows with `stride` elements between rows, on the device.  When shard_depth > 0 the first
// shard_depth levels of the split are applied to all n_all points and only subtree shard_index is kept and built
// (pn_build_opts.shard_depth / shard_index); *n_out receives its size and `shape` its tree shape.  `alloc_out` is
// called once n_out and the shape are known and must return the output arrays.  Returns 0 or a cudaError_t value;
// err receives the detail.
template <typename A>
int build_ball_tree(const A* raw, uint64_t n_all, uint32_t d, uint64_t stride, uint32_t bucket_size, uint32_t shard_depth,
                    uint32_t shard_index, TreeShape& shape, uint64_t* n_out,
                    BallOut<A> (*alloc_out)(void* ctx, uint64_t n, const TreeShape& shape), void* ctx, cudaStream_t st,
                    std::string& err, uint32_t rule = 0, uint32_t order_levels = 0);
// rule 0: the reference's split (the first column with the greatest spread, src/ball_tree.rs:577-613) -- the layout the host
//         builder produces, bit for bit.
// rule 1: the TWO-MEANS split (not the reference's; an engine-internal partition for the pruned tensor scan): the key of a
//         point is its projection on the line through the two centroids of a 2-means clustering of a sample of its
//         segment; median cut, shape, centroids and radii as for rule 0, so every query path is exact on the result.
//         `order_levels` more levels of the same split order the rows inside the buckets.

// ---- vantage-point tree (src/vantage_point_tree.rs:146-197): ranges of the level-l slices in the stored order; the
// vantage point of a slice [lo, hi) sits at hi - 1, near = [lo, lo + (len-1)/2), far = [lo + (len-1)/2, hi - 1)
struct VpShape {
    uint64_t n = 0;
    uint32_t L = 0;
    std::vector<std::vector<uint32_t>> lo, hi;  // [L + 1][2^l]
    void init(uint64_t n_, uint32_t L_);
};
template <typename A>
struct VpOut {
    A* pts;            // n x dpad, stored order [near | far | vantage point] recursively, buckets sorted by (distance to the parent's vantage point, id)
    uint32_t* ids;     // n
    A* centers;        // n_internal x dpad: vantage point rows
    A* radii;          // n_internal: mu
    uint32_t* vp_ids;  // n_internal
};
template <typename A>
int build_vp_tree(const A* raw, uint64_t n, uint32_t d, uint64_t stride, uint32_t bucket_size, VpShape& shape,
                  VpOut<A> (*alloc_out)(void* ctx, uint64_t n, const VpShape& shape), void* ctx, cudaStream_t st, std::string& err);

// mean of the stored rows (double accumulation over fixed chunks of 4096 rows combined in chunk order: the same value
// as the host pass of DeviceTree::prepare_tensor) and the largest centred coordinate max |p_j - c_j|
int centre_and_range_f32(const float* pts, uint64_t n, uint32_t d, uint32_t dpad, float* center_dev, float* center_host,
                         float* maxabs, cudaStream_t st, std::string& err);

}  // namespace gb
}  // namespace petal
