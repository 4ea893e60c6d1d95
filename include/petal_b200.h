/*
 * petal_b200.h -- C ABI of libpetal_b200.so, the B200-native (sm_100a) exact nearest-neighbour
 * engine behind the petal-neighbors API.
 *
 * The reference (petabi/petal-neighbors v0.18.0) is a pure-Rust library with no FFI of its
 * own; its public Rust API is the drop-in surface and this header is what a Rust `extern "C"`
 * block (rust/petal-neighbors-b200/src/ffi.rs, shown in INTEGRATION.md) binds underneath it.
 * Every entry point names the reference interface it replaces (file:line into the reference).
 *
 * Conventions
 *   - plain pointers and sizes only; no C++/torch types cross the boundary;
 *   - every function returns a pn_status (int32_t); pn_last_error_message() gives the
 *     thread-local detail string; no exception or panic crosses the ABI;
 *   - `A` is f32 or f64 (the reference is generic over `A: Float`), one symbol per type;
 *   - host-buffer calls (`pn_*_query_*`) copy queries H2D and results D2H themselves;
 *     `_dev` calls take device pointers on the tree's device and enqueue on `stream`;
 *   - indices are u64 at the boundary (Rust `usize`), u32 inside the engine (N < 2^32);
 *   - k-NN results are ordered by (distance, index) ascending -- the reference's order for
 *     distinct distances, with index as the tie-break (BASELINE.json north_star); rows are
 *     padded with (UINT64_MAX, +inf) when k > n;
 *   - distances are bit-identical to the reference's sequential non-FMA fold + sqrt
 *     (src/distance.rs:26-35);
 *   - there is no CPU fallback: a query on a machine without a usable CUDA device fails with
 *     PN_CUDA.
 * Threading: queries on one tree from several host threads are legal (the reference's
 * `&self` queries, `Euclidean: Sync`, src/distance.rs:19); on one handle they serialise on an
 * internal mutex, on sessions of it (pn_tree_session) they run concurrently.  create/destroy
 * must not race with queries on the same handle.
 */
#ifndef PETAL_B200_H
#define PETAL_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PN_ABI_VERSION 1

typedef enum pn_status {
    PN_OK = 0,
    PN_EMPTY = 1,          /* ArrayError::Empty,         src/lib.rs:12-13, src/ball_tree.rs:44-46 */
    PN_NOT_CONTIGUOUS = 2, /* ArrayError::NotContiguous, src/lib.rs:14-15, src/ball_tree.rs:47-49 */
    PN_BAD_ARG = 3,        /* null pointer, dtype/kind mismatch, n >= 2^32, bad option */
    PN_CUDA = 4,           /* CUDA runtime error or no device (no CPU fallback) */
    PN_NCCL = 5,           /* NCCL could not be loaded, or a collective failed (pn_comm_*, pn_sharded_*, pn_tree_replicate) */
    PN_OOM = 6             /* host or device allocation failed */
} pn_status;

typedef enum pn_tree_kind { PN_KIND_BALL = 0, PN_KIND_VP = 1 } pn_tree_kind;
typedef enum pn_dtype { PN_F32 = 0, PN_F64 = 1 } pn_dtype;

/* scan engine selection for k-NN */
typedef enum pn_algo {
    PN_ALGO_AUTO = 0,
    PN_ALGO_SIMT = 1,  /* exact difference-form FP32/FP64 tiles on the CUDA cores */
    PN_ALGO_TENSOR = 2 /* tcgen05 FP16 filter + exact rerank (f32 input; AUTO: every batch size when d >= 16) */
} pn_algo;

/* Where the tree is built.  Both builders apply the reference's split rule and produce bit-identical flattened
 * layouts (points of a bucket in ascending original index); AUTO builds on the device when the tree has a device
 * and at least 32768 points.  (BASELINE.json: "tree construction stays on the host" -- the host builder remains
 * the default for small trees and the checker of the device builder; SURVEY.md 8f row 2.) */
typedef enum pn_builder { PN_BUILDER_AUTO = 0, PN_BUILDER_HOST = 1, PN_BUILDER_DEVICE = 2 } pn_builder;

/* Pruning of (query group, point tile) pairs on the tensor path (k <= 16): AUTO turns it on when a build-time estimate
 * says at least a quarter of those pairs are out of reach (clustered data); uniform data in d >= 16 prunes nothing and
 * skips the set-up passes.  Results are identical either way. */
typedef enum pn_prune { PN_PRUNE_AUTO = 0, PN_PRUNE_ON = 1, PN_PRUNE_OFF = 2 } pn_prune;

/* Which partition of the points the tensor path scans (k-NN batches of f32 trees with d >= 16).  Exact results do not depend
 * on it; what the tile bitmaps of the pruned scan can skip does.  REFERENCE: the tree's own stored order (the reference's
 * split: median of the widest coordinate, src/ball_tree.rs:577-613).  TWO_MEANS: the handle also keeps a second ball tree
 * over the same rows whose splits follow the line through the two centroids of a 2-means clustering of each node -- buckets
 * follow clusters instead of cutting through them -- and answers k-NN batches from it.  AUTO builds it where the build-time
 * estimates say seeding pays but the reference partition's tile balls are too loose, and keeps it when its own estimates
 * turn the tile bitmaps on (clustered data in d >= 32, e.g. BASELINE config 3); uniform data never pays for it.  The
 * layout accessors, self-queries and radius queries of a ball handle always use the reference partition. */
typedef enum pn_partition { PN_PARTITION_AUTO = 0, PN_PARTITION_REFERENCE = 1, PN_PARTITION_TWO_MEANS = 2 } pn_partition;

#define PN_FLAG_HOST_ONLY 1u /* build + flatten on the host only (no device; queries fail with
                                PN_CUDA).  For builder tests on machines without a GPU. */

/* Engine knobs.  The reference has none (SURVEY.md 5); all are new.  Zero = default. */
typedef struct pn_build_opts {
    uint32_t struct_size; /* sizeof(pn_build_opts), for forward compatibility */
    int32_t device;       /* CUDA device ordinal; -1 = current device */
    uint32_t bucket_size; /* target points per leaf bucket (default 256, min 8) */
    uint32_t algo;        /* pn_algo */
    uint32_t host_threads; /* builder threads; 0 = hardware concurrency */
    uint32_t flags;
    /* Point sharding by subtree (multi-GPU, "points larger than one GPU's HBM"): keep only the
     * points of subtree `shard_index` at depth `shard_depth` of the ball tree
     * (src/ball_tree.rs:535-537 split rule).  Returned indices stay global.  0/0 = all. */
    uint32_t shard_depth;
    uint32_t shard_index;
    uint32_t builder;     /* pn_builder: where the partition is computed */
    uint32_t prune;       /* pn_prune: triangle-inequality pruning in front of the tensor filter */
    uint32_t partition;   /* pn_partition: the partition the tensor path scans */
    uint32_t reserved[5];
} pn_build_opts;

typedef struct pn_tree pn_tree; /* opaque: flattened, device-resident tree */

typedef struct pn_tree_info {
    uint64_t n_points;     /* points held by this handle (shard-local) */
    uint64_t n_points_total;
    uint32_t dim, dim_padded;
    uint32_t kind, dtype;
    uint32_t n_levels;     /* cut level L: buckets are the reference's nodes at depth L */
    uint32_t n_buckets, n_nodes;
    uint32_t bucket_size_max;
    int32_t device;
    uint32_t algo;
    uint64_t device_bytes;
    double build_seconds;  /* build + flatten + upload + tensor-path set-up */
    /* pruning decisions of the tensor path and the build-time estimates behind them (0 when the tensor path is off) */
    uint32_t prune_seeded;      /* queries are sorted by home bucket and start from a seed threshold */
    uint32_t prune_tiles;       /* per-CTA tile bitmaps are computed and tiles skipped */
    double est_seed_candidates; /* candidates a query still reranks when it starts from its seed */
    double est_tile_frac;       /* share of tile balls beyond a single query's seed */
    double est_group_tile_frac; /* share of tile balls out of reach of a whole tile of queries */
    uint32_t tensor_partition;  /* the partition the estimates above describe and k-NN batches scan: 0 reference, 1 two-means */
    uint32_t reserved0;
} pn_tree_info;

/* Work counters of the most recent query call (SURVEY.md 8d). */
typedef struct pn_counters {
    uint64_t queries;
    uint64_t pairs;          /* (query, point) distances evaluated by the scan kernels */
    uint64_t filter_pairs;   /* (query, point) pairs seen by the tensor filter */
    uint64_t rerank_pairs;   /* candidates re-evaluated exactly after the tensor filter */
    uint64_t node_visits;    /* (query tile, node) visits of the traversal */
    uint64_t kernel_launches;
    double device_ms;        /* CUDA-event time of the device work of the call */
    double scan_ms;          /* CUDA-event time of the dominant (scan/filter) kernel alone */
    uint64_t h2d_bytes, d2h_bytes;
} pn_counters;

const char *pn_last_error_message(void);
int32_t pn_abi_version(void);
int32_t pn_device_count(int32_t *count);

/* --- construction: BallTree::new / ::euclidean (src/ball_tree.rs:38-63, 367-373) and
 * VantagePointTree::new / ::euclidean (src/vantage_point_tree.rs:31-72).  `points` is row-major
 * with `row_stride` elements between rows and `col_stride` between the elements of a row
 * (col_stride != 1 -> PN_NOT_CONTIGUOUS, the reference's row-0 check).  The buffer is borrowed
 * for the duration of the call only.  `opts` may be NULL. */
int32_t pn_balltree_create_f32(const float *points, size_t n, size_t d, size_t row_stride,
                               size_t col_stride, const pn_build_opts *opts, pn_tree **out);
int32_t pn_balltree_create_f64(const double *points, size_t n, size_t d, size_t row_stride,
                               size_t col_stride, const pn_build_opts *opts, pn_tree **out);
int32_t pn_vptree_create_f32(const float *points, size_t n, size_t d, size_t row_stride,
                             size_t col_stride, const pn_build_opts *opts, pn_tree **out);
int32_t pn_vptree_create_f64(const double *points, size_t n, size_t d, size_t row_stride,
                             size_t col_stride, const pn_build_opts *opts, pn_tree **out);
/* The same for points that already live on the device `opts->device` (row-major, unit column stride): the partition
 * is computed on the GPU (src/ball_tree.rs:445-613 level by level) and nothing crosses PCIe. */
int32_t pn_balltree_create_dev_f32(const float *points_dev, size_t n, size_t d, size_t row_stride,
                                   const pn_build_opts *opts, pn_tree **out);
int32_t pn_balltree_create_dev_f64(const double *points_dev, size_t n, size_t d, size_t row_stride,
                                   const pn_build_opts *opts, pn_tree **out);
int32_t pn_tree_destroy(pn_tree *tree); /* Rust Drop */

/* --- sessions: concurrent callers.  The reference's queries take `&self` and `Euclidean` is `Sync`
 * (src/distance.rs:19), so several threads may query one tree at once.  Calls on ONE handle serialise on its mutex
 * (they share one stream and one set of workspaces).  A session is a second handle onto the same device-resident tree
 * -- nothing of the tree is copied -- with its own stream, events, workspaces and counters: calls on different
 * sessions overlap on the device.  One session per calling thread is the intended use.  The tree, including a
 * partition built later by a query on any of them, is shared by the handle and all its sessions (and their sessions)
 * and lives until the last of them is destroyed, in any order.  Its device memory is reported by the handle that built
 * it (pn_tree_info::device_bytes; 0 on a session).  A session answers every query entry point of its tree's kind. */
int32_t pn_tree_session(pn_tree *tree, pn_tree **out);

/* --- BallTree::query (src/ball_tree.rs:102-121), batched: `nq` queries, row stride
 * `q_row_stride` elements; outputs are caller-allocated row-major nq x k.  k == 0 is a no-op
 * (:106-108). */
int32_t pn_balltree_query_f32(pn_tree *tree, const float *queries, size_t nq, size_t q_row_stride,
                              size_t k, uint64_t *idx_out, float *dist_out);
int32_t pn_balltree_query_f64(pn_tree *tree, const double *queries, size_t nq, size_t q_row_stride,
                              size_t k, uint64_t *idx_out, double *dist_out);

/* --- BallTree::query_nearest (src/ball_tree.rs:80-86), batched; outputs nq each. */
int32_t pn_balltree_query_nearest_f32(pn_tree *tree, const float *queries, size_t nq,
                                      size_t q_row_stride, uint64_t *idx_out, float *dist_out);
int32_t pn_balltree_query_nearest_f64(pn_tree *tree, const double *queries, size_t nq,
                                      size_t q_row_stride, uint64_t *idx_out, double *dist_out);

/* --- BallTree::query_radius (src/ball_tree.rs:137-142), batched.  Result is CSR:
 * offsets[nq + 1], indices[offsets[nq]] (strict `distance < r` on the bit-exact distance,
 * :277; each query's indices ascending).  Both arrays are engine-allocated; release each with
 * pn_free. */
int32_t pn_balltree_query_radius_f32(pn_tree *tree, const float *queries, size_t nq,
                                     size_t q_row_stride, float radius, uint64_t **offsets_out,
                                     uint64_t **indices_out);
int32_t pn_balltree_query_radius_f64(pn_tree *tree, const double *queries, size_t nq,
                                     size_t q_row_stride, double radius, uint64_t **offsets_out,
                                     uint64_t **indices_out);

/* --- VantagePointTree::query_nearest (src/vantage_point_tree.rs:88-98), batched. */
int32_t pn_vptree_query_nearest_f32(pn_tree *tree, const float *queries, size_t nq,
                                    size_t q_row_stride, uint64_t *idx_out, float *dist_out);
int32_t pn_vptree_query_nearest_f64(pn_tree *tree, const double *queries, size_t nq,
                                    size_t q_row_stride, uint64_t *idx_out, double *dist_out);

/* --- k-NN and radius search on a vantage-point handle (SURVEY.md 8f row 4).  EXTENSIONS: the reference's
 * VantagePointTree has query_nearest only (src/vantage_point_tree.rs:88-98).  The results are those BallTree::query /
 * BallTree::query_radius return for the same points (same (distance, index) order, same strict `< r`, same output
 * shapes as pn_balltree_query_* above): exact answers do not depend on the partition.  k-NN runs on the vantage-point
 * arrays (or, for tensor-eligible trees, on the ball partition the handle keeps next to them); radius search on a ball
 * partition of the stored points, built on the device at the first such call. */
int32_t pn_vptree_query_f32(pn_tree *tree, const float *queries, size_t nq, size_t q_row_stride,
                            size_t k, uint64_t *idx_out, float *dist_out);
int32_t pn_vptree_query_f64(pn_tree *tree, const double *queries, size_t nq, size_t q_row_stride,
                            size_t k, uint64_t *idx_out, double *dist_out);
int32_t pn_vptree_query_radius_f32(pn_tree *tree, const float *queries, size_t nq,
                                   size_t q_row_stride, float radius, uint64_t **offsets_out,
                                   uint64_t **indices_out);
int32_t pn_vptree_query_radius_f64(pn_tree *tree, const double *queries, size_t nq,
                                   size_t q_row_stride, double radius, uint64_t **offsets_out,
                                   uint64_t **indices_out);

/* --- all-points self-query: every stored point is a query (the reference bench's loop,
 * benches/ball_tree.rs:53-59, and the k-NN-graph shape of downstream clustering).  Row i of the
 * n x k outputs is the answer for points[i]; the point itself is its own first neighbour
 * (distance 0, lowest index among exact duplicates).  No query upload: the stored, bucket-ordered
 * points are the query tiles.  pn_tree_query_self_dev is the same call into device buffers (n x k on the tree's
 * device; `stream` and `sync` as for pn_tree_query_knn_dev below).  It takes any handle of a whole tree -- ball or
 * vantage-point tree, or a session of either -- and gives the same rows on each; a handle that holds one shard of a
 * tree (shard_depth > 0) returns PN_BAD_ARG. */
int32_t pn_balltree_query_self_f32(pn_tree *tree, size_t k, uint64_t *idx_out, float *dist_out);
int32_t pn_balltree_query_self_f64(pn_tree *tree, size_t k, uint64_t *idx_out, double *dist_out);
int32_t pn_tree_query_self_dev(pn_tree *tree, size_t k, uint64_t *idx_dev, void *dist_dev, void *stream,
                               int32_t sync);

/* --- distance::pairwise with the Euclidean metric (src/distance.rs:58-74): dense symmetric n x n
 * matrix of exact distances, zero diagonal; `out` is caller-allocated row-major n x n host memory.
 * (A "next" row of the scope table: not on the tree path, same bit-exact fold.) */
int32_t pn_pairwise_f32(int32_t device, const float *x, size_t n, size_t d, size_t row_stride, float *out);
int32_t pn_pairwise_f64(int32_t device, const double *x, size_t n, size_t d, size_t row_stride, double *out);

void pn_free(void *p);

/* --- device-resident variants (queries and outputs already in HBM on the tree's device).
 * Used by the bench's kernel-only leg and by multi-GPU drivers that all-gather per-shard
 * results.  `stream` is a cudaStream_t (NULL = the tree's own stream); the call returns after
 * enqueueing unless `sync` != 0.  The element type is the tree's dtype. */
int32_t pn_tree_query_knn_dev(pn_tree *tree, const void *queries_dev, size_t nq,
                              size_t q_row_stride, size_t k, uint64_t *idx_dev, void *dist_dev,
                              void *stream, int32_t sync);

/* Radius search from and into device memory: the result of pn_balltree_query_radius_* / pn_vptree_query_radius_* (strict
 * `distance < r` on the bit-exact distance, each query's indices ascending) as CSR in caller buffers on the tree's device.
 * - The element type of queries_dev is the tree's dtype; `radius` is converted to it (exact for any value of that type).
 * - Any handle: a ball or vantage-point tree (a VP tree answers from its ball partition, as its radius call does), a
 *   session of either, or a handle of one shard (shard_depth > 0), whose indices are global.
 * - offsets_dev[nq + 1] is always written in full and equals the offsets the host call returns; offsets_dev[nq] is the
 *   total.  offsets_dev == NULL is PN_BAD_ARG.  nq == 0 writes offsets_dev[0] = 0.
 * - Query q's segment is written to indices_dev[offsets[q] .. offsets[q + 1]) if and only if offsets[q + 1] <= capacity;
 *   nothing is ever written at or past `capacity`.  The offsets do not decrease, so the written queries are a prefix of
 *   the batch: a caller whose buffer was too small reads the total, then reallocates or re-issues only the queries after
 *   that prefix.  indices_dev may be NULL only with capacity == 0 (offsets only).
 * - Argument checks as pn_tree_query_knn_dev: a PN_FLAG_HOST_ONLY handle returns PN_CUDA; nq < 2^32; q_row_stride >= d
 *   when nq > 1.
 * - `stream` NULL is the handle's own stream.  With sync == 0 the call returns after enqueueing: no stream, event or device
 *   synchronisation and no device-to-host copy happens inside, except that (1) the first radius call on a VP handle
 *   may build its ball partition (f64, d < 16 or fewer than 1024 points); (2) a call on another stream than the
 *   handle's previous call first waits for that stream, as for k-NN; (3) the workspaces are sized per chunk of
 *   queries (the whole batch up to 2^18 queries, otherwise chunks of 2^17), and a call whose chunk is larger than that
 *   of every earlier radius call on the handle allocates larger ones -- freeing and allocating device memory can
 *   synchronise the device, as for k-NN.  Once the workspaces are warm, the guarantee holds without exception.  With
 *   sync != 0 the call waits, and the counters (pairs, device_ms, ...) describe it. */
int32_t pn_tree_query_radius_dev(pn_tree *tree, const void *queries_dev, size_t nq, size_t q_row_stride,
                                 double radius, uint64_t *offsets_dev, uint64_t *indices_dev, size_t capacity,
                                 void *stream, int32_t sync);

/* K-way merge of `n_lists` per-shard sorted top-k lists (layout [list][nq][k]) by
 * (distance, index): the step after the all-gather when points are sharded by subtree
 * (no reference equivalent; SURVEY.md 8e).  All pointers are device pointers on `device`. */
int32_t pn_merge_topk_dev(uint32_t dtype, int32_t device, const uint64_t *idx_lists_dev,
                          const void *dist_lists_dev, size_t n_lists, size_t nq, size_t k,
                          uint64_t *idx_out_dev, void *dist_out_dev, void *stream, int32_t sync);

/* Merge of n_lists per-shard CSR radius results over the same nq queries (the step after the exchange when points are
 * sharded by subtree; no reference equivalent).  offsets_lists_dev[n_lists][nq + 1] are absolute positions into
 * indices_lists_dev; each list's segment of a query is ascending.  out_offsets_dev[nq + 1]; out_indices_dev holds
 * sum over lists of (offsets[l][nq] - offsets[l][0]) entries.  Equal indices from different lists are kept, in list
 * order.  All pointers are device pointers on `device`. */
int32_t pn_merge_radius_dev(int32_t device, const uint64_t *offsets_lists_dev, const uint64_t *indices_lists_dev,
                            size_t n_lists, size_t nq, uint64_t *out_offsets_dev, uint64_t *out_indices_dev,
                            void *stream, int32_t sync);

/* --- multi-GPU inside the library (SURVEY.md 8e; no reference equivalent: the crate is single-threaded).
 * A pn_comm is ONE RANK of an NCCL communicator bound to one device.  One process per GPU: rank 0 calls
 * pn_comm_unique_id, the host language ships the 128 bytes to the other ranks (MPI, torch.distributed, a file ...), every
 * rank calls pn_comm_create.  One process driving several GPUs: pn_comm_create_all makes all ranks at once
 * (ncclCommInitAll); calls that communicate must then be issued from one host thread per rank.
 * NCCL is loaded at run time (libnccl.so.2; PN_NCCL_LIB overrides), so single-GPU users never need it. */
typedef struct pn_comm pn_comm;
#define PN_UNIQUE_ID_BYTES 128
int32_t pn_comm_unique_id(void *id_out);
int32_t pn_comm_create(const void *unique_id, int32_t world, int32_t rank, int32_t device, pn_comm **out);
int32_t pn_comm_create_all(const int32_t *devices, int32_t n_dev, pn_comm **out /* n_dev entries */);
int32_t pn_comm_destroy(pn_comm *comm);

/* How the per-shard lists meet. */
typedef enum pn_exchange {
    PN_EXCHANGE_ALLGATHER = 0, /* ncclAllGather: every rank ends with the merged result of ALL queries */
    PN_EXCHANGE_SLICE = 1      /* grouped ncclSend/ncclRecv: rank r ends with the merged rows of ITS query slice only
                                  (world x less traffic); slice r = pn_query_slice(nq, r, world) */
} pn_exchange;

typedef struct pn_shard_stats {
    double scan_ms;      /* sum over chunks: local tensor/SIMT scan + packing, CUDA events on the compute stream */
    double exchange_ms;  /* sum over chunks: the NCCL calls, CUDA events on the exchange stream (overlaps the next scan) */
    double merge_ms;     /* sum over chunks: k-way merge kernels (PEER exchange: end of this rank's last scan to the end of its last merge) */
    double total_ms;     /* first enqueue to last merge */
    uint64_t nccl_bytes_sent; /* payload bytes this rank sent to OTHER ranks */
    uint64_t nccl_calls;
    uint64_t rows_out;   /* result rows written on this rank */
    uint32_t n_chunks;
    uint32_t peer_mib;   /* PEER exchange: MiB this rank's merge kernels read from other devices' memory */
} pn_shard_stats;

/* contiguous slice [*lo, *hi) of a batch of nq queries owned by `rank` (sizes differ by at most one) */
void pn_query_slice(size_t nq, int32_t rank, int32_t world, size_t *lo, size_t *hi);

/* Point sharding by subtree: `tree` holds subtree `rank` at depth log2(world) (pn_build_opts.shard_depth / shard_index),
 * `queries_dev` holds ALL nq queries on this rank's device (the same on every rank).  Every rank scans its shard in
 * chunks of queries; the sorted per-shard lists of chunk i (8-byte (distance, index) keys for f32) cross NVLink through
 * NCCL on the exchange stream while chunk i+1 is scanned, and a k-way merge kernel produces the final rows:
 * all nq rows on every rank (ALLGATHER), or the rows of this rank's slice, idx/dist_dev sized for the slice (SLICE).
 * k <= 255.  Collective: every rank of `comm` must make the same call. */
int32_t pn_sharded_query_knn_dev(pn_tree *tree, pn_comm *comm, const void *queries_dev, size_t nq,
                                 size_t q_row_stride, size_t k, uint32_t exchange, uint64_t *idx_dev,
                                 void *dist_dev, void *stream, pn_shard_stats *stats);

/* Query sharding with the tree replicated: the flattened tree of `root` (all device arrays, including the tensor-path
 * operand image) is sent to every other rank with ncclBroadcast instead of being rebuilt there.  On `root`, `tree` is the
 * source and *out = tree; elsewhere `tree` is NULL and *out receives a new handle.  Collective. */
int32_t pn_tree_replicate(pn_tree *tree, pn_comm *comm, int32_t root, pn_tree **out);

/* --- one process driving several GPUs: the survey's pn_ctx.  A pn_multi owns one rank per device (ncclCommInitAll),
 * one host thread per rank for every call, and either a replica of the tree on every device (PN_SHARD_REPLICATE: built
 * once on the first device, sent to the others with ncclBroadcast; a batch of queries is split into contiguous slices,
 * no data-path collective) or one subtree per device (PN_SHARD_BY_SUBTREE: n_dev a power of two; every device scans all
 * queries on its shard, lists exchanged slice-wise over NCCL and merged on the owning device).  Host buffers in and out,
 * same result layout and semantics as pn_balltree_query_*.  This is what a Rust or C++ host calls to use a whole box
 * through the C ABI. */
typedef struct pn_multi pn_multi;
typedef enum pn_shard_mode { PN_SHARD_REPLICATE = 0, PN_SHARD_BY_SUBTREE = 1 } pn_shard_mode;
int32_t pn_multi_balltree_create_f32(const int32_t *devices, int32_t n_dev, uint32_t shard_mode, const float *points,
                                     size_t n, size_t d, size_t row_stride, const pn_build_opts *opts, pn_multi **out);
int32_t pn_multi_balltree_query_f32(pn_multi *m, const float *queries, size_t nq, size_t q_row_stride, size_t k,
                                    uint64_t *idx_out, float *dist_out);
/* Radius search on a multi-GPU handle: the CSR result pn_balltree_query_radius_f32 returns on a tree of all the points
 * (strict distance < r, each query's indices ascending), engine-allocated, released with pn_free.
 * REPLICATE: every device answers its slice of the batch.  BY_SUBTREE: every device answers all queries on its shard, the
 * owner of each slice pulls the shards' hit lists of its slice with peer copies (no NCCL; pn_multi_set_exchange applies to
 * k-NN only) and merges them on its device.  Each slice is written straight into its region of the single result. */
int32_t pn_multi_balltree_query_radius_f32(pn_multi *m, const float *queries, size_t nq, size_t q_row_stride,
                                           float radius, uint64_t **offsets_out, uint64_t **indices_out);
/* How the per-shard lists of a BY_SUBTREE handle meet: PN_EXCHANGE_PEER (the default when every pair of devices has peer
 * access) runs NO collective -- the k-way merge kernel of each device reads the other devices' packed lists directly from
 * their memory over NVLink (the exchange fused into the consumer); PN_EXCHANGE_SLICE uses grouped ncclSend/ncclRecv. */
#define PN_EXCHANGE_PEER 2u
int32_t pn_multi_set_exchange(pn_multi *m, uint32_t exchange);
/* per-device statistics of the last query: stats[n_dev] (BY_SUBTREE: the exchange; REPLICATE: zeros but rows_out).  After a
 * radius search: scan_ms = traversal, exchange_ms = peer pulls, merge_ms = counts + offsets scan + merge, total_ms, rows_out,
 * n_chunks (traversal chunks), peer_mib = MiB pulled from other devices; no NCCL calls. */
int32_t pn_multi_get_stats(const pn_multi *m, pn_shard_stats *stats, int32_t n_stats);
int32_t pn_multi_destroy(pn_multi *m);

/* --- introspection */
int32_t pn_tree_get_info(const pn_tree *tree, pn_tree_info *info);
int32_t pn_tree_get_counters(const pn_tree *tree, pn_counters *counters);

/* Copy-out of the flattened layout (builder tests; SURVEY.md 7 step 3).  Any pointer may be
 * NULL.  ids[n]: original index of the i-th point in bucket order; bucket_lo/hi[n_buckets];
 * node_radius[n_nodes] (ball: radius, vp: threshold mu); node_center[n_nodes * dim_padded]
 * (ball: centroid, vp: vantage point); points[n * dim_padded] in the tree's dtype. */
int32_t pn_tree_get_layout(const pn_tree *tree, uint32_t *ids, uint32_t *bucket_lo,
                           uint32_t *bucket_hi, void *node_radius, void *node_center,
                           void *points);

#ifdef __cplusplus
}
#endif
#endif /* PETAL_B200_H */
