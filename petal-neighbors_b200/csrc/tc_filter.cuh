// tc_filter.cuh -- tensor-core k-NN scan: tcgen05 FP16 filter + exact difference-form rerank.
//
// Where the query x bucket tile really is a dense contraction (f32, d >= 16: the ball bounds
// prune nothing, pairs/(N*Q) ~ 1), the distance matrix is evaluated on the 5th-gen tensor cores as
//     D~^2(q,p) = |q'|^2 + |p'|^2 - 2 q'.p'      (q' = s (q - c), p' = s (p - c); c = data mean,
//                                                  s = power of two with max |p'_j| <= 1)
// by ONE augmented FP16 contraction (fp32 accumulate): A row = [q'_0 .. q'_{d-1}, n1, n2, n3, 1, 1, 1,
// 0..] with |q'|^2 = n1+n2+n3 split into fp16 pieces, B row = [-2p'_0 .., 1, 1, 1, m1, m2, m3, 0..], so
// the TMEM accumulator holds D~^2 itself and the epilogue is a bare threshold test (the K steps of 16 that
// hold nothing but the zero padding are never issued).  FP16
// has the significand of TF32 at half the bytes (L2->SM operand traffic and shared-memory operand
// reads both halve).
// The filter is only a filter: every element with D~^2 <= Theta_q is re-evaluated with the exact
// sequential non-FMA fold of kernels.cuh (Euclidean::distance, reference src/distance.rs:26-35)
// and selected on the (sqrt'd distance, index) key, so results are bit-identical to the SIMT path
// and the oracle.
//
// Theta_q = s^2 thresh2(kth_q) (1 + (d+4) 2^-23) + E_q with the rigorous rounding bound (scaled units)
//   E_q = 1.01 2^-9 |q'| Pmax + 2^-14 sqrt(d) (|q'| + 2 Pmax) + (Kp+8) 2^-21 (|q'| + Pmax)^2
// (round-to-nearest fp16 inputs: 2^-11 relative per factor; 2^-14 absolute per coordinate covers the
// subnormal range even if the tensor core flushed fp16 denormals;
// three-piece norms: < 2^-30; fp32 accumulation, norm evaluation and centring: the quadratic term).
// Queries whose scaled norm leaves the fp16 range get E_q = +inf: every point is reranked exactly.
//
// Structure (one CTA = MT x 128 queries, persistent over its share of the point tiles; 1 CTA / SM;
// MT x NUM_ACC x SW = the 512 TMEM columns: 2 subtiles x 2 stages x 128 for wide rows, 4 x 1 x 128 for two or three
// K chunks, 4 x 2 x 64 -- half-tile stages -- for one K chunk):
//   warps 4MT, 5MT+1 : two producers on alternate ring groups: 1-D bulk copies (cp.async.bulk) of the
//                pre-tiled, pre-swizzled B image ([128 rows x 32 fp16] chunks, 64B swizzle)
//   warps 4MT+1.. : MT tcgen05.mma issuers, one per 128-query subtile: the whole warp runs the loop on
//                warp-uniform values, elect.sync picks the issuing lane (descriptors stay in uniform
//                registers); kind::f16, M=128 N=128 K=16 per instruction
//   warps 0..4MT-1 : epilogue, one query row per thread: tcgen05.ld 32x32b.x32 -> stage released ->
//                    FMNMX3 min tree -> threshold -> ballot-compacted hit queue -> batched exact rerank
//                    + sorted insertion into the owning thread's top-k (shared memory)
// grid.y splits the point stream (small batches, the last partial wave of large ones); the splits of a
// query share their k-th bounds through global memory and merge_lists_kernel merges their lists.
// Seeds and pruning (tc_prune.cuh): a query may start from a seed threshold instead of +inf (FilterArgs::seed_t2), and
// the PRUNE instantiation scans only the tiles of the CTA's bitmap, every role walking the bitmap on its own.
#pragma once
#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "kernels.cuh"
#include "tc_prune.cuh"

namespace petal {
namespace tc {

// -DPN_TC_PROFILE: per-role cycle accounting into counters[8..] (diagnostic builds only)
#ifdef PN_TC_PROFILE
// 32-bit clocks and accumulators: the roles run with as few as 80 registers per thread
#define PROF_DECL unsigned pt_ = (unsigned)clock(), pc_[6] = {0, 0, 0, 0, 0, 0}
#define PROF_ADD(i) do { unsigned n_ = (unsigned)clock(); pc_[i] += n_ - pt_; pt_ = n_; } while (0)
#define PROF_FLUSH(base) do { for (int i_ = 0; i_ < 6; ++i_) atomicAdd(&a.counters[8 + (base) + i_], (unsigned long long)pc_[i_]); } while (0)
#else
#define PROF_DECL
#define PROF_ADD(i)
#define PROF_FLUSH(base)
#endif
// -DPN_TC_TRACE (with PN_TC_PROFILE): timeline trace of CTA 0: trace[(role * 64 + (tile - trace_t0)) * 4 + event] = clock64()
#if defined(PN_TC_PROFILE) && defined(PN_TC_TRACE)
#define TRACE(role, tile, ev) do { if (a.trace && blockIdx.x == 0 && (tile) >= a.trace_t0 && (tile) < a.trace_t0 + 64u) a.trace[(((role) * 64) + ((tile) - a.trace_t0)) * 4 + (ev)] = clock64(); } while (0)
#else
#define TRACE(role, tile, ev)
#endif

constexpr int BM = 128;            // queries per accumulator tile (TMEM lanes)
constexpr int BN = 128;            // points per B tile (TMEM columns per accumulator stage)
constexpr int KC = 32;             // fp16 elements per K chunk = one 64-byte swizzle row
constexpr int CHUNK_BYTES = BN * KC * 2;   // 8 KB: one B ring slot
constexpr int A_CHUNK_BYTES = BM * KC * 2; // 8 KB: one resident A chunk
constexpr int NSLOT = 6;           // K slots used by the folded norms

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// Blocking wait.  The suspend-time hint lets the hardware put the waiting thread to sleep until the
// phase completes (wake-up ~60 cycles) instead of re-issuing try_wait in a tight loop: the spinning
// producer / MMA-issuer lanes share schedulers with epilogue warps and, being the highest warp ids,
// would otherwise win arbitration and starve them.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred P1;\n\t"
        "WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1, %2;\n\t"
        "@P1 bra DONE;\n\t"
        "bra WAIT_LOOP;\n\t"
        "DONE:\n\t"
        "}" ::"r"(smem_u32(bar)), "r"(parity), "r"(1000000u) : "memory");
}
__device__ __forceinline__ void tma_load_2d(const CUtensorMap* map, uint64_t* bar, void* dst, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
            smem_u32(dst)),
        "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void bulk_copy(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
// true on exactly one lane of a fully converged warp; unlike `lane == 0` it keeps every value computed
// from warp-uniform inputs in the uniform datapath, so tcgen05.mma gets its descriptors straight from
// uniform registers (a per-thread branch makes ptxas wrap every UTCHMMA in an ELECT / R2UR.BROADCAST
// loop, and each issue then waits ~250 cycles for the previous one: scripts/mma_rate.cu)
__device__ __forceinline__ bool elect_one() {
    uint32_t pred = 0;
    asm volatile("{\n\t.reg .pred px;\n\telect.sync _|px, 0xffffffff;\n\tselp.u32 %0, 1, 0, px;\n\t}" : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// D[tmem] (+)= A[smem] * B[smem], kind::f16 (fp16 inputs, fp32 accumulate), both operands K-major
__device__ __forceinline__ void tc_mma_f16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(d_tmem),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// same, A operand from tensor memory (TS form): [lane = query row][K packed two fp16 per 32-bit column]
__device__ __forceinline__ void tc_mma_f16_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t"
        "}" ::"r"(d_tmem),
        "r"(a_tmem), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// shared memory -> tensor memory copy of one K step of the A operand: 128 rows x 256 bits (16 fp16) = 8 columns
__device__ __forceinline__ void tc_cp_128x256b(uint32_t taddr, uint64_t sdesc) {
    asm volatile("tcgen05.cp.cta_group::1.128x256b [%0], %1;" ::"r"(taddr), "l"(sdesc) : "memory");
}
// K-major, 64-byte swizzle shared-memory matrix descriptor (cute::UMMA::SmemDescriptor layout):
// start>>4 [0,14) | LBO>>4 = 1 [16,30) | SBO>>4 = (8 rows x 64 B)/16 [32,46) | version 1 [46,48) | SWIZZLE_64B = 4 [61,64)
__device__ __forceinline__ uint64_t make_desc_sw64(uint32_t saddr) {
    return (uint64_t)((saddr >> 4) & 0x3FFF) | (1ull << 16) | (32ull << 32) | (1ull << 46) | (4ull << 61);
}
// kind::f16 instruction descriptor: D=F32 [4,6)=1, A=B=F16 [7,10)=[10,13)=0, K-major both, N>>3 [17,23), M>>4 [24,29)
__host__ __device__ constexpr uint32_t make_idesc_f16(int M, int N) {
    return (1u << 4) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// asynchronous TMEM load of 32 consecutive columns of this thread's lane; the registers are valid
// only after tmem_ld_wait(), which takes them as in/out operands so nothing is scheduled across it
__device__ __forceinline__ void tmem_ld32_issue(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait(uint32_t (&r)[32]) {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "+r"(r[8]),
                   "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15]), "+r"(r[16]),
                   "+r"(r[17]), "+r"(r[18]), "+r"(r[19]), "+r"(r[20]), "+r"(r[21]), "+r"(r[22]), "+r"(r[23]), "+r"(r[24]),
                   "+r"(r[25]), "+r"(r[26]), "+r"(r[27]), "+r"(r[28]), "+r"(r[29]), "+r"(r[30]), "+r"(r[31])
                 :
                 : "memory");
}

// three-input min (FMNMX3); NaN inputs drop out as in fminf.  Written in PTX: from nested fminf the compiler forms
// two-input mins of the columns first and spends 38 instructions on 64 columns instead of 32.
__device__ __forceinline__ float min3f(float a, float b, float c) {
    float d;
    asm("min.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c));
    return d;
}
// Minimum of a 64-column accumulator unit with 31 three-input mins and one two-input min, as one chain: it keeps a
// single partial minimum live next to the 64 columns, which the hit search still needs (the epilogue runs at 80
// registers).  The result is <= theta iff some column is (a NaN column never is).
__device__ __forceinline__ float unit_min64(const uint32_t (&r)[2][32]) {
    float acc = min3f(__uint_as_float(r[0][0]), __uint_as_float(r[0][1]), __uint_as_float(r[0][2]));
#pragma unroll
    for (int c = 3; c < 63; c += 2) acc = min3f(acc, __uint_as_float(r[c / 32][c % 32]), __uint_as_float(r[(c + 1) / 32][(c + 1) % 32]));
    return fminf(acc, __uint_as_float(r[1][31]));
}
// the same wait for the two 32-column groups of a 64-column unit: one tcgen05.wait::ld covers every load issued before it
__device__ __forceinline__ void tmem_ld_wait(uint32_t (&r)[2][32]) {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(r[0][0]), "+r"(r[0][1]), "+r"(r[0][2]), "+r"(r[0][3]), "+r"(r[0][4]), "+r"(r[0][5]), "+r"(r[0][6]), "+r"(r[0][7]),
                   "+r"(r[0][8]), "+r"(r[0][9]), "+r"(r[0][10]), "+r"(r[0][11]), "+r"(r[0][12]), "+r"(r[0][13]), "+r"(r[0][14]), "+r"(r[0][15]),
                   "+r"(r[0][16]), "+r"(r[0][17]), "+r"(r[0][18]), "+r"(r[0][19]), "+r"(r[0][20]), "+r"(r[0][21]), "+r"(r[0][22]), "+r"(r[0][23]),
                   "+r"(r[0][24]), "+r"(r[0][25]), "+r"(r[0][26]), "+r"(r[0][27]), "+r"(r[0][28]), "+r"(r[0][29]), "+r"(r[0][30]), "+r"(r[0][31]),
                   "+r"(r[1][0]), "+r"(r[1][1]), "+r"(r[1][2]), "+r"(r[1][3]), "+r"(r[1][4]), "+r"(r[1][5]), "+r"(r[1][6]), "+r"(r[1][7]),
                   "+r"(r[1][8]), "+r"(r[1][9]), "+r"(r[1][10]), "+r"(r[1][11]), "+r"(r[1][12]), "+r"(r[1][13]), "+r"(r[1][14]), "+r"(r[1][15]),
                   "+r"(r[1][16]), "+r"(r[1][17]), "+r"(r[1][18]), "+r"(r[1][19]), "+r"(r[1][20]), "+r"(r[1][21]), "+r"(r[1][22]), "+r"(r[1][23]),
                   "+r"(r[1][24]), "+r"(r[1][25]), "+r"(r[1][26]), "+r"(r[1][27]), "+r"(r[1][28]), "+r"(r[1][29]), "+r"(r[1][30]), "+r"(r[1][31])
                 :
                 : "memory");
}
// Per-thread running top-k kept in SHARED memory ([slot][lane], conflict-free): it is only touched
// when the hit queue is drained, and keeping it out of the register file lets the epilogue hold a
// whole accumulator stage in registers instead.  Only the k-th key / thresh2 live in registers.
// Same (distance, index) order and floor semantics as TopK in kernels.cuh.  An entry is ONE 64-bit key,
// (float bits of the sqrt'd distance) << 32 | index: distances are non-negative, so unsigned integer order of the
// key is exactly the lexicographic (distance, index) order, an empty slot (+inf, NO_ID) is the largest key, and a
// shift of the sorted insertion is one 64-bit load, one compare and one 64-bit store.  (The hit path is bound by
// instruction issue in divergent code -- an insertion with independent loads but more instructions was 1.6x slower.)
struct SmemTopK {
    unsigned long long* sk;  // [k][32] keys of this warp, this lane's column = lane
    unsigned long long kth_key, floor_key;
    float t2;
    uint32_t k;
    static __device__ __forceinline__ unsigned long long make_key(float d, uint32_t i) {
        return ((unsigned long long)__float_as_uint(d) << 32) | i;
    }
    __device__ __forceinline__ void init(unsigned long long* base, int lane, uint32_t k_, bool active) {
        sk = base + lane; k = k_;
        kth_key = make_key(pos_inf<float>(), NO_ID);
        for (uint32_t s = 0; s < k; ++s) sk[s * 32] = kth_key;
        t2 = active ? pos_inf<float>() : -1.f;
        floor_key = 0ull;  // nothing is below it: set_floor() raises it
    }
    __device__ __forceinline__ void set_floor(float d, uint32_t i) { floor_key = make_key(d, i) + 1ull; }  // keys must exceed (d, i)
    __device__ __forceinline__ bool offer_key(unsigned long long key) {
        if (key < floor_key || key >= kth_key) return false;
        uint32_t p = k - 1;  // sorted insertion from the tail
        while (p > 0) {
            const unsigned long long pk = sk[(p - 1) * 32];
            if (key >= pk) break;
            sk[p * 32] = pk;
            --p;
        }
        sk[p * 32] = key;
        kth_key = sk[(k - 1) * 32];
        t2 = thresh2(__uint_as_float((uint32_t)(kth_key >> 32)));
        return true;
    }
    __device__ __forceinline__ void store(float* out_d, uint32_t* out_i) const {
        for (uint32_t s = 0; s < k; ++s) {
            const unsigned long long e = sk[s * 32];
            out_d[s] = __uint_as_float((uint32_t)(e >> 32)); out_i[s] = (uint32_t)e;
        }
    }
};

struct FilterArgs {
    DevTree<float> t;
    const float4* q;       // nq x dpad exact zero-padded queries (rerank)
    const float* q_margin; // nq: E_q in scaled units (+inf when the query leaves the fp16 range)
    uint32_t nq, k;        // nq: one past the last query row of this launch
    uint32_t row0;         // first query row of this launch (CTA x serves rows row0 + x MT 128 ...)
    uint32_t n_tiles;      // ceil(n / BN)
    uint32_t tiles_per_split;  // grid.y splits the point stream: CTA (x, y) scans tiles [y tps, min(n_tiles, (y+1) tps))
                               // and writes list y; the lists are merged by merge_lists_kernel
    uint32_t nkc;          // K chunks (Kp / 32)
    uint32_t last_steps;   // K steps of 16 that the last chunk really holds (1 or 2): (d + 6) mod 32 in 1..16 -> 1
    uint32_t stages;       // B ring depth in groups
    uint32_t gs;           // chunks per ring group (one full/empty barrier pair per group)
    float t2_scale;        // s^2 (1 + (d+4) 2^-23): exact squared threshold -> scaled filter units
    float* g_bound;        // [nq - row0] or null: k-th bounds (exact squared units) shared by the splits of a query
    float* part_d;         // [grid.y][nq - row0][k]
    uint32_t* part_i;
    const float* floor_d;
    const uint32_t* floor_i;
    unsigned long long* counters;  // [2] filter hits (elements passed to the exact rerank)
    // pruned scan (tc_prune.cuh): CTA x scans only the tiles whose bit is set in its bitmap, and every query starts from
    // its seed threshold
    const uint32_t* tile_bits;     // [grid.x][tile_words]
    const uint32_t* tile_cnt;      // [grid.x] set bits
    const float* seed_t2;          // [nq] or null: thresh2 of the seed k-th distance (exact squared units); also used by the dense scan
    uint32_t tile_words;
#ifdef PN_TC_PROFILE
    uint32_t dbg;          // diagnostic leg isolation: 1 = epilogue skips the scan, 2 = producer skips the copies
    long long* trace;      // optional timeline of CTA 0, 12 roles x 64 tiles x 4 events
    uint32_t trace_t0;
#endif
};

// three-piece fp16 split of a non-negative fp32 value (residual < 2^-30 x in the normal range)
__device__ __forceinline__ void split3_f16(float x, __half& h1, __half& h2, __half& h3) {
    h1 = __float2half_rn(x);
    const float r1 = x - __half2float(h1);
    h2 = __float2half_rn(r1);
    h3 = __float2half_rn(r1 - __half2float(h2));
}

// B operand: one fp16 row per stored point (bucket order), written as the exact shared-memory image
// the MMA reads: [tile of 128 points][K chunk of 32 fp16][128 rows x 64 B, 64-byte swizzle], so one
// ring group is ONE contiguous span of global memory and is fetched by a single 1-D bulk copy (a
// tensor-map request of 128 separate 64-byte rows kept the per-SM feed at ~10 B/cycle).
// 64-byte swizzle: the 16-byte unit index (address bits 4-5) is XORed with address bits 7-8 = (row >> 1) & 3.
// pmax_bits receives max |p'| (float bits).  The buffer is zero-filled first (rows past n).
__device__ __forceinline__ size_t baug_offset(uint32_t row, uint32_t j, uint32_t nkc) {
    const uint32_t tile = row / BN, r = row % BN, c = j / KC, e = j % KC;
    return ((size_t)(tile * nkc + c) * BN + r) * KC + (((e >> 3) ^ ((r >> 1) & 3u)) << 3) + (e & 7u);
}
__global__ void build_baug_kernel(const float* __restrict__ pts, const float* __restrict__ center, float scale, uint32_t n,
                                  uint32_t d, uint32_t dpad, uint32_t kp, __half* __restrict__ baug, unsigned int* pmax_bits) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float* p = pts + (size_t)i * dpad;
    const uint32_t nkc = kp / KC;
    float nrm = 0.f;
    for (uint32_t j = 0; j < d; ++j) {
        const float v = (p[j] - center[j]) * scale;
        nrm = nrm + v * v;
        baug[baug_offset(i, j, nkc)] = __float2half_rn(-2.0f * v);
    }
    // the six norm slots follow the data dimensions directly (K = d .. d+5) and the zero padding comes last, so that the
    // K steps of 16 that hold nothing but padding are never issued (d = 128: 9 MMAs per tile instead of 10)
    for (uint32_t j = d + NSLOT; j < kp; ++j) baug[baug_offset(i, j, nkc)] = __float2half_rn(0.f);
    __half h1, h2, h3;
    split3_f16(nrm, h1, h2, h3);
    const __half one = __float2half_rn(1.f);
    baug[baug_offset(i, d, nkc)] = one;     baug[baug_offset(i, d + 1, nkc)] = one; baug[baug_offset(i, d + 2, nkc)] = one;
    baug[baug_offset(i, d + 3, nkc)] = h1;  baug[baug_offset(i, d + 4, nkc)] = h2;  baug[baug_offset(i, d + 5, nkc)] = h3;
    atomicMax(pmax_bits, __float_as_uint(sqrtf(nrm) * 1.000001f));
}

// A operand + per-query margin E_q (scaled units)
__global__ void build_aaug_kernel(const float* __restrict__ q, const float* __restrict__ center, float scale, uint32_t nq,
                                  uint32_t d, uint32_t dpad, uint32_t kp, float pmax, __half* __restrict__ aaug,
                                  float* __restrict__ q_margin) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nq) return;
    const float* p = q + (size_t)i * dpad;
    __half* o = aaug + (size_t)i * kp;
    float nrm = 0.f;
    for (uint32_t j = 0; j < d; ++j) {
        const float v = (p[j] - center[j]) * scale;
        nrm = nrm + v * v;
    }
    const float qn = sqrtf(nrm) * 1.000001f;
    const bool in_range = qn <= 200.f;  // every coordinate and the norm stay finite in fp16
    for (uint32_t j = 0; j < d; ++j) o[j] = __float2half_rn(in_range ? (p[j] - center[j]) * scale : 0.f);
    for (uint32_t j = d + NSLOT; j < kp; ++j) o[j] = __float2half_rn(0.f);
    __half h1, h2, h3;
    split3_f16(in_range ? nrm : 0.f, h1, h2, h3);
    const __half one = __float2half_rn(1.f);
    o[d] = h1; o[d + 1] = h2; o[d + 2] = h3; o[d + 3] = one; o[d + 4] = one; o[d + 5] = one;
    const float sn = qn + pmax;
    const float e = 1.01f * 0.001953125f * qn * pmax + 6.2e-05f * sqrtf((float)d) * (qn + 2.f * pmax) +
                    (float)(kp + 8) * 4.76837158203125e-07f * sn * sn;
    q_margin[i] = in_range ? e : pos_inf<float>();
}

// MT subtiles of 128 queries per CTA, NUM_ACC accumulator stages per subtile (MT x NUM_ACC x 128 = the 512 TMEM
// columns).  Wide rows (tensor-pipe bound) run MT = 2 x NUM_ACC = 2.  Narrow rows (d <= 58), where the epilogue
// is the bound and each warp's wait -> read-out -> test -> push chain is latency-bound, run MT = 4 x NUM_ACC = 1:
// sixteen epilogue warps, four independent chains per scheduler, and the tensor pipe round-robins over the four
// subtiles so that one subtile's read-out hides behind the other three's MMAs.  With 22 warps the register
// file allows 93 registers per thread, so a stage is read out and tested in two halves of 64 columns.
// SHARED: the launch splits the point stream (grid.y > 1) and the splits of a query share their k-th bounds; compiled
// out of the whole-stream launch, where the extra state costs registers the 80-register configuration does not have.
template <int DVR, int K, int MT, int NUM_ACC, bool SHARED, int SW = BN, bool PRUNE = false>
__global__ void __launch_bounds__((5 * MT + 2) * 32, 1)
knn_filter_kernel(const __grid_constant__ CUtensorMap map_a, const unsigned char* __restrict__ baug, const FilterArgs a) {
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    // carve: [A: MT*nkc chunks][B ring: stages chunks][barriers]
    unsigned char* smem = (unsigned char*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    unsigned char* smem_a = smem;
    unsigned char* smem_b = smem + (size_t)MT * a.nkc * A_CHUNK_BYTES;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem_b + (size_t)a.stages * a.gs * CHUNK_BYTES);
    uint64_t* full_bar = bars;                       // [stages]
    uint64_t* empty_bar = bars + a.stages;           // [stages]
    uint64_t* tfull_bar = bars + 2 * a.stages;       // [NUM_ACC][MT]
    uint64_t* tempty_bar = tfull_bar + NUM_ACC * MT; // [NUM_ACC][MT]
    uint64_t* a_bar = tempty_bar + NUM_ACC * MT;     // [1]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(a_bar + 1);
    uint32_t* qbuf = tmem_slot + 4;  // per epilogue warp: QWORDS x u32 of queue / hand-over scratch
    constexpr int QWORDS = 192;  // 64 queue entries + 32 hand-over slots, 8 bytes each
    unsigned long long* tk = reinterpret_cast<unsigned long long*>(qbuf + 4 * MT * QWORDS);   // [EPI_WARPS][k][32] keys, k = a.k <= K

    const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0), lane = threadIdx.x & 31;  // warp-uniform for the compiler
    constexpr int EPI_WARPS = 4 * MT;
    // Wide rows with one accumulator stage per subtile keep the A operand in tensor memory (TS-form MMA): the pipe then
    // reads only B from shared memory (measured 70 instead of 85 cycles per 128x128x16 MMA, scripts/mma_rate.cu).
    // Columns: MT accumulators of 128, then MT A operands of Kp/2 (two fp16 per column), 512 allocated.
    // With half-tile stages (SW = 64) the two subtiles keep TWO accumulator stages each next to their A operands:
    // 2 x 2 x 64 accumulator columns + 2 x nkc x 16 operand columns <= 512 up to nkc = 8.
    // THREE subtiles x one whole-tile stage (384 columns) leave 128 columns: three operands of up to five K steps
    // (8 columns each), i.e. rows of up to 74 dimensions.
    constexpr bool TS = (MT == 2 && (NUM_ACC == 1 || SW == 64)) || MT == 3;
    constexpr int TMEM_COLS = TS ? 512 : NUM_ACC * MT * SW;  // power of two
    // accumulator units per B tile: a stage holds SW columns, i.e. the distances of 128 queries to SW of the tile's 128
    // points; with SW = 64 the four-subtile configuration gets TWO stages per subtile out of the same 512 columns
    constexpr int U = BN / SW;
    static_assert(SW == BN || SW == 64, "stage width is a whole tile or half a tile");

    if (warp == EPI_WARPS && lane == 0) {
        for (uint32_t s = 0; s < a.stages; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], MT); }
        for (int s = 0; s < NUM_ACC * MT; ++s) { mbar_init(&tfull_bar[s], 1); mbar_init(&tempty_bar[s], 4); }
        mbar_init(a_bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_a) : "memory");
    }
    if (warp == EPI_WARPS + 1) {  // first MMA warp owns the TMEM allocation
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);

    const uint32_t row_base = a.row0 + blockIdx.x * (MT * BM);
    // this CTA's share of the point stream (every split is non-empty: the host guarantees grid.y tps < n_tiles + tps)
    // (pruned scan: the set bits of this CTA's tile bitmap instead, walked by every role on its own)
    static_assert(!(PRUNE && SHARED), "the pruned scan does not split the point stream");
    const uint32_t j_begin = PRUNE ? 0u : blockIdx.y * a.tiles_per_split;
    const uint32_t n_my = PRUNE ? a.tile_cnt[blockIdx.x] : min(a.n_tiles - j_begin, a.tiles_per_split);
    const uint32_t* my_bits = PRUNE ? a.tile_bits + (size_t)blockIdx.x * a.tile_words : nullptr;

    if (warp == EPI_WARPS || warp == EPI_WARPS + MT + 1) {
        // ================= TMA producers: two warps, alternate ring groups (stages is even) =================
        const uint32_t pid = warp == EPI_WARPS ? 0u : 1u;
        if (lane == 0) {
            if (pid == 0) {
                mbar_expect_tx(a_bar, (uint32_t)(MT * a.nkc * A_CHUNK_BYTES));
                for (int mt = 0; mt < MT; ++mt)
                    for (uint32_t c = 0; c < a.nkc; ++c)
                        tma_load_2d(&map_a, a_bar, smem_a + (size_t)(mt * a.nkc + c) * A_CHUNK_BYTES, (int)(c * KC), (int)(row_base + mt * BM));
            }
            // B ring: groups of `gs` chunks share one full/empty barrier pair, so the consumers pay one
            // barrier wait per group instead of one per 8 KB chunk
            const uint32_t total = n_my * a.nkc;
            const uint32_t n_groups = (total + a.gs - 1) / a.gs;
            const unsigned char* bsrc = baug + (size_t)j_begin * a.nkc * CHUNK_BYTES;
            PROF_DECL;
            if (PRUNE) {
                // the tiles of the list are not contiguous in the image: one bulk copy per 8 KB chunk, the chunks of a ring
                // group still complete on the group's one barrier
                TileIter it;
                if (n_my) it.init(my_bits);
                for (uint32_t i = 0, ch = 0; i < n_my; ++i) {
                    const uint32_t tile = it.next();
                    for (uint32_t c = 0; c < a.nkc; ++c, ++ch) {
                        const uint32_t g = ch / a.gs, gi = ch % a.gs;
                        if ((g & 1u) != pid) continue;
                        const uint32_t s = g % a.stages, ph = (g / a.stages) & 1u;
                        if (gi == 0) {
                            mbar_wait(&empty_bar[s], ph ^ 1u);
                            mbar_expect_tx(&full_bar[s], min(a.gs, total - ch) * CHUNK_BYTES);
                        }
                        bulk_copy(smem_b + (size_t)(s * a.gs + gi) * CHUNK_BYTES, baug + ((size_t)tile * a.nkc + c) * CHUNK_BYTES, CHUNK_BYTES, &full_bar[s]);
                    }
                }
            } else
            for (uint32_t g = pid; g < n_groups; g += 2) {
                const uint32_t s = g % a.stages, ph = (g / a.stages) & 1u;
                const uint32_t first = g * a.gs, cnt = min(a.gs, total - first);
                PROF_ADD(1);
                mbar_wait(&empty_bar[s], ph ^ 1u);
                PROF_ADD(0);
#ifdef PN_TC_PROFILE
                if (a.dbg & 2u) { mbar_arrive(&full_bar[s]); continue; }
#endif
                // chunk `it` of the stream sits at byte it * CHUNK_BYTES of the tiled image: one contiguous span per group
                mbar_expect_tx(&full_bar[s], cnt * CHUNK_BYTES);
                bulk_copy(smem_b + (size_t)s * a.gs * CHUNK_BYTES, bsrc + (size_t)first * CHUNK_BYTES, cnt * CHUNK_BYTES, &full_bar[s]);
            }
            if (pid == 0) PROF_FLUSH(12);
        }
    } else if (warp > EPI_WARPS && warp <= EPI_WARPS + MT) {
        // ================= MMA issuers: one warp (one elected lane) per 128-query subtile ==========
        // The issuing thread's serial chain of mbarrier waits (~90 cycles each even when complete)
        // and tcgen05.mma issues is what bounds small-K tiles, so it is split over MT threads.
        // The whole warp runs the loop on warp-uniform values; one elected lane issues.
        {
            const int mt = warp - (EPI_WARPS + 1);
            const uint64_t a_desc0 = make_desc_sw64(smem_u32(smem_a)) + (uint64_t)(mt * a.nkc * (A_CHUNK_BYTES >> 4));
            const uint64_t b_desc0 = make_desc_sw64(smem_u32(smem_b));
            const uint32_t total = n_my * a.nkc;
            mbar_wait(a_bar, 0);
            // TS: this subtile's A operand goes to tensor memory once, K step by K step (copies and MMAs issued by one
            // thread execute in order)
            const uint32_t a_ksteps = 2 * a.nkc - (a.last_steps > 1 ? 0u : 1u);   // K steps of 16 that carry data
            const uint32_t a_tmem = tmem_base + NUM_ACC * MT * SW + mt * (a_ksteps * 8);
            if (TS) {
                tc_fence_after();
                if (elect_one()) {
                    for (uint32_t c = 0; c < a.nkc; ++c) {
                        const uint64_t ad = a_desc0 + (uint64_t)(c * (A_CHUNK_BYTES >> 4));
                        tc_cp_128x256b(a_tmem + c * 16, ad);
                        if (c + 1 < a.nkc || a.last_steps > 1) tc_cp_128x256b(a_tmem + c * 16 + 8, ad + 2);
                    }
                }
                __syncwarp();
            }
            uint32_t it = 0, g = 0, gi = 0, s = 0, sph = 0;  // stream position: group, chunk in group, ring stage, its phase
            uint32_t u = 0;  // accumulator units issued so far: stage u % NUM_ACC, phase (u / NUM_ACC) & 1
            constexpr uint32_t idesc_u = make_idesc_f16(BM, SW);
            PROF_DECL;
            for (uint32_t j = 0; j < n_my; ++j) {
                const uint32_t it0 = it, g0 = g, gi0 = gi, s0 = s, sph0 = sph;  // ring position of this tile's first chunk
#pragma unroll
                for (int h = 0; h < U; ++h, ++u) {
                    // every unit of a tile walks the tile's chunks again (rows [h SW, (h+1) SW) of each); the ring
                    // groups are waited for by the first unit and handed back by the last
                    if (h) { it = it0; g = g0; gi = gi0; s = s0; sph = sph0; }
                    const uint32_t as = u % NUM_ACC, aph = (u / NUM_ACC) & 1u;
                    mbar_wait(&tempty_bar[as * MT + mt], aph ^ 1u);  // this subtile's accumulator stage has been read out
                    tc_fence_after();
                    PROF_ADD(0);
                    if (lane == 0) TRACE(8 + mt, j, 0);
                    const uint32_t d_tmem = tmem_base + (as * MT + mt) * SW;
                    for (uint32_t c = 0; c < a.nkc; ++c, ++it) {
                        if (gi == 0 && h == 0) {
                            mbar_wait(&full_bar[s], sph);
                            tc_fence_after();
                            PROF_ADD(1);
                        }
                        if (lane == 0 && c == 0) TRACE(8 + mt, j, 1);
                        // descriptors advance in 16-byte units: +2 per K step of 16 fp16, whole chunks per slot, 64 B per row
                        const uint64_t bd = b_desc0 + (uint64_t)((s * a.gs + gi) * (CHUNK_BYTES >> 4) + h * (SW * KC * 2 >> 4));
                        const uint64_t ad = a_desc0 + (uint64_t)(c * (A_CHUNK_BYTES >> 4));
                        const bool last = gi + 1 == a.gs || it + 1 == total;
                        if (elect_one()) {
                            const bool two = c + 1 < a.nkc || a.last_steps > 1;  // the upper half of the last chunk may be padding only
                            if (TS) {
                                tc_mma_f16_ts(d_tmem, a_tmem + c * 16, bd, idesc_u, c > 0 ? 1u : 0u);
                                if (two) tc_mma_f16_ts(d_tmem, a_tmem + c * 16 + 8, bd + 2, idesc_u, 1u);
                            } else {
                                tc_mma_f16(d_tmem, ad, bd, idesc_u, c > 0 ? 1u : 0u);
                                if (two) tc_mma_f16(d_tmem, ad + 2, bd + 2, idesc_u, 1u);
                            }
                            if (last && h == U - 1) tc_commit(&empty_bar[s]);  // group consumed by this subtile
                        }
                        __syncwarp();
                        if (last) { gi = 0; ++g; if (++s == a.stages) { s = 0; sph ^= 1u; } } else ++gi;
                    }
                    if (elect_one()) tc_commit(&tfull_bar[as * MT + mt]);  // this unit's accumulator is complete
                    __syncwarp();
                    PROF_ADD(2);
                    if (lane == 0) TRACE(8 + mt, j, 2);
                }
            }
            if (mt == 0 && lane == 0) PROF_FLUSH(0);
        }
    } else {
        // ================= epilogue: one query row per thread =================
        // Filter hits are not evaluated in place (a divergent chain of dependent L2 round trips
        // that would hold the accumulator stage hostage for the whole CTA): they are pushed to a
        // per-warp queue with ballot compaction and drained 32 at a time, the 32 lanes evaluating
        // 32 exact distances in parallel and handing each result to the lane that owns the query.
        const int mt = warp >> 2, quad = warp & 3;
        const uint32_t wrow0 = row_base + mt * BM + quad * 32;  // first query row of this warp
        const uint32_t qrow = wrow0 + lane;
        const bool active = qrow < a.nq;
        const DevTree<float>& t = a.t;
        const int DV = DVR > 0 ? DVR : (int)t.dv;
        // per-warp scratch: 64 queued point rows, 64 owner lanes, 32 + 32 hand-over slots
        // per-warp scratch: 64 queue entries (point row | owner lane << 32) and 32 hand-over slots (top-k keys)
        unsigned long long* q_ent = reinterpret_cast<unsigned long long*>(qbuf + warp * QWORDS);
        unsigned long long* x_key = q_ent + 64;
        SmemTopK topk;
        topk.init(tk + warp * (a.k * 32), lane, a.k, active);
        if (a.floor_d && active) topk.set_floor(a.floor_d[qrow], a.floor_i[qrow]);
        const float margin = active ? a.q_margin[qrow] : 0.f;  // E_q (scaled units)
        const float t2s = a.t2_scale;
        const float seed2 = a.seed_t2 && active ? a.seed_t2[qrow] : pos_inf<float>();  // an upper bound of the final k-th distance
        TileIter titer;
        if (PRUNE && n_my) titer.init(my_bits);
        float theta = active ? xadd(xmul(seed2, t2s), margin) : -pos_inf<float>();   // +inf without a seed
        // Theta_q from the best known k-th bound.  When the point stream is split over several CTAs, the k-th distance
        // of ANY split's list is an upper bound of the final k-th distance, so the splits of a query publish theirs
        // (atomicMin on the float bits: the bounds are non-negative) and each filters with the smallest one.
        float* gb = SHARED && active ? a.g_bound + (qrow - a.row0) : nullptr;
        auto refresh_theta = [&](bool publish) {
            float b = fminf(topk.t2, seed2);
            if (SHARED && gb) {
                if (publish) atomicMin(reinterpret_cast<int*>(gb), __float_as_int(b));
                b = fminf(b, __ldcg(gb));
            }
            theta = xadd(xmul(b, t2s), margin);
        };
        const unsigned full = 0xffffffffu;
        const unsigned lt_mask = (1u << lane) - 1u;
        unsigned long long hits = 0;
        int qn = 0;  // queue fill, warp-uniform

        // exact evaluation of queue entries [0, cnt), cnt <= 32 (warp-uniform): lane e evaluates entry
        // e; results are handed to the owning lanes in rounds (one entry per owner per round) so all
        // owners insert concurrently
        auto drain = [&](int cnt) {
            unsigned long long key = ~0ull;
            int o = 32 + lane;  // unique dummy owner for idle lanes
            const bool valid = lane < cnt;
            if (valid) {
                const unsigned long long e = q_ent[lane];
                o = (int)(e >> 32);
                const uint32_t prow = (uint32_t)e;
                const float4* qr = a.q + (size_t)(wrow0 + o) * DV;
                const float4* pr = t.pts + (size_t)prow * DV;
                float acc = 0.f;
                if (DVR > 0) {
#pragma unroll
                    for (int jc = 0; jc < (DVR > 0 ? DVR : 1); ++jc) acc = fold(acc, __ldg(qr + jc), __ldg(pr + jc));
                } else {
                    for (int jc = 0; jc < DV; ++jc) acc = fold(acc, __ldg(qr + jc), __ldg(pr + jc));
                }
                // the evaluating lanes take the square roots in parallel; the owners only compare and insert keys
                key = SmemTopK::make_key(xsqrt(acc), __ldg(t.ids + prow));
            }
            const unsigned grp = __match_any_sync(full, o);
            const int rank = __popc(grp & lt_mask);
            const int rounds = __reduce_max_sync(full, valid ? rank + 1 : 0);
            for (int r = 0; r < rounds; ++r) {
                const bool send = valid && rank == r;
                if (send) x_key[o] = key;
                const unsigned owners = __reduce_or_sync(full, send ? (1u << o) : 0u);
                __syncwarp();
                if ((owners >> lane) & 1u) {
                    if (topk.offer_key(x_key[lane])) refresh_theta(true);
                }
                __syncwarp();
            }
        };

        // threshold test of 32 accumulator columns [col0, col0+32) of tile j: per-lane hit mask in `bits`; returns
        // (warp-uniform) whether any lane of the warp has a hit
        auto test32 = [&](const uint32_t (&r)[32], uint32_t j, int col0, uint32_t& bits) -> bool {
            // block minima over 4 blocks of 8 consecutive columns; only blocks that pass are searched
            float mb[4];
#pragma unroll
            for (int b = 0; b < 4; ++b) {
                const float x0 = fminf(__uint_as_float(r[8 * b]), fminf(__uint_as_float(r[8 * b + 1]), __uint_as_float(r[8 * b + 2])));
                const float x1 = fminf(__uint_as_float(r[8 * b + 3]), fminf(__uint_as_float(r[8 * b + 4]), __uint_as_float(r[8 * b + 5])));
                mb[b] = fminf(fminf(x0, x1), fminf(__uint_as_float(r[8 * b + 6]), __uint_as_float(r[8 * b + 7])));
            }
            const float m = fminf(fminf(mb[0], mb[1]), fminf(mb[2], mb[3]));
            bits = 0;
            if (!__any_sync(full, m <= theta)) return false;
            if (m <= theta) {
#pragma unroll
                for (int b = 0; b < 4; ++b) {
                    if (mb[b] <= theta) {
#pragma unroll
                        for (int i = 0; i < 8; ++i) bits |= (__uint_as_float(r[8 * b + i]) <= theta ? 1u : 0u) << (8 * b + i);
                    }
                }
                const int valid = (int)t.n - (int)(j * BN + col0);  // rows past the last point are zero-filled
                if (valid < 32) bits &= valid > 0 ? ((1u << valid) - 1u) : 0u;
            }
            return true;
        };
        // hits of one 32-column group go to the warp's queue (ballot compaction); a full queue is drained at once
        auto push32 = [&](uint32_t bits, uint32_t j, int col0) {
            for (;;) {
                const bool has = bits != 0;
                const unsigned mask = __ballot_sync(full, has);
                if (!mask) break;
                if (has) {
                    const int i = __ffs(bits) - 1;
                    bits &= bits - 1;
                    const int slot = qn + __popc(mask & lt_mask);
                    const uint32_t prow = j * BN + col0 + i;
                    q_ent[slot] = (unsigned long long)prow | ((unsigned long long)lane << 32);
                    // the exact rerank happens tiles later: start pulling the candidate's row and id now
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(t.pts + (size_t)prow * DV));
                }
                qn += __popc(mask);
                hits += __popc(mask);
                __syncwarp();
                if (qn >= 32) {
                    drain(32);
                    const int rest = qn - 32;  // < 32
                    unsigned long long te = 0;
                    if (lane < rest) te = q_ent[32 + lane];
                    __syncwarp();
                    if (lane < rest) q_ent[lane] = te;
                    __syncwarp();
                    qn = rest;
                }
            }
        };

        // fused threshold test + push of one group (two-stage configurations): a threshold tightened by a drain
        // already applies to the next group of the same tile
        auto scan32 = [&](const uint32_t (&r)[32], uint32_t j, int col0) {
            // block minima over 4 blocks of 8 consecutive columns; only blocks that pass are searched
            float mb[4];
#pragma unroll
            for (int b = 0; b < 4; ++b) {
                const float x0 = fminf(__uint_as_float(r[8 * b]), fminf(__uint_as_float(r[8 * b + 1]), __uint_as_float(r[8 * b + 2])));
                const float x1 = fminf(__uint_as_float(r[8 * b + 3]), fminf(__uint_as_float(r[8 * b + 4]), __uint_as_float(r[8 * b + 5])));
                mb[b] = fminf(fminf(x0, x1), fminf(__uint_as_float(r[8 * b + 6]), __uint_as_float(r[8 * b + 7])));
            }
            const float m = fminf(fminf(mb[0], mb[1]), fminf(mb[2], mb[3]));
            if (!__any_sync(full, m <= theta)) return;
            uint32_t bits = 0;
            if (m <= theta) {
#pragma unroll
                for (int b = 0; b < 4; ++b) {
                    if (mb[b] <= theta) {
#pragma unroll
                        for (int i = 0; i < 8; ++i) bits |= (__uint_as_float(r[8 * b + i]) <= theta ? 1u : 0u) << (8 * b + i);
                    }
                }
                const int valid = (int)t.n - (int)(j * BN + col0);  // rows past the last point are zero-filled
                if (valid < 32) bits &= valid > 0 ? ((1u << valid) - 1u) : 0u;
            }
            for (;;) {
                const bool has = bits != 0;
                const unsigned mask = __ballot_sync(full, has);
                if (!mask) break;
                if (has) {
                    const int i = __ffs(bits) - 1;
                    bits &= bits - 1;
                    const int slot = qn + __popc(mask & lt_mask);
                    const uint32_t prow = j * BN + col0 + i;
                    q_ent[slot] = (unsigned long long)prow | ((unsigned long long)lane << 32);
                    // the exact rerank happens tiles later: start pulling the candidate's row and id now
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(t.pts + (size_t)prow * DV));
                }
                qn += __popc(mask);
                hits += __popc(mask);
                __syncwarp();
                if (qn >= 32) {
                    drain(32);
                    const int rest = qn - 32;  // < 32
                    unsigned long long te = 0;
                    if (lane < rest) te = q_ent[32 + lane];
                    __syncwarp();
                    if (lane < rest) q_ent[lane] = te;
                    __syncwarp();
                    qn = rest;
                }
            }
        };

        // The whole 128-column accumulator stage is pulled into registers at once and released
        // BEFORE it is tested: with only two stages in TMEM the MMA -> read-out -> release loop of a
        // stage is the critical path, so nothing but the TMEM loads may sit inside it.
        if constexpr (MT <= 2 && SW == BN) {
            constexpr int G = BN / 32;
            uint32_t r[G][32];
            const uint32_t lane_off = (uint32_t)(quad * 32) << 16;
            PROF_DECL;
            for (uint32_t jr = 0; jr < n_my; ++jr) {
                const uint32_t j = PRUNE ? titer.next() : j_begin + jr;  // absolute tile (point rows); stage and phase follow the CTA's own count
                const uint32_t as = jr % NUM_ACC, aph = (jr / NUM_ACC) & 1u;
                PROF_ADD(3);
                mbar_wait(&tfull_bar[as * MT + mt], aph);
                tc_fence_after();
                PROF_ADD(0);
                const uint32_t taddr = tmem_base + lane_off + (as * MT + mt) * BN;
    #pragma unroll
                for (int g = 0; g < G; ++g) tmem_ld32_issue(taddr + g * 32, r[g]);
    #pragma unroll
                for (int g = 0; g < G; ++g) tmem_ld_wait(r[g]);
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&tempty_bar[as * MT + mt]);
                PROF_ADD(1);
    #ifdef PN_TC_PROFILE
                if (a.dbg & 1u) continue;
    #endif
    #pragma unroll
                for (int g = 0; g < G; ++g) scan32(r[g], j, g * 32);
                PROF_ADD(2);
                // scheduled drain: every warp of the CTA drains in the same tile, so the stalls coincide
                if (((PRUNE ? jr : j) & 31u) == 31u) {
                    if (qn > 0) { drain(qn); qn = 0; __syncwarp(); }
                    if (SHARED && gb) refresh_theta(false);  // pick up the other splits' progress
                }
            }
            if (warp == 0 && lane == 0) PROF_FLUSH(6);
        } else if constexpr (SW < BN) {
            // Half-tile stages (narrow rows): each subtile owns TWO 64-column stages, so the MMA of the next half tile runs
            // while this one is read out and tested, and the four warps sharing a stage get half a tile of slack against
            // each other (with one whole-tile stage the slowest sibling's hit path gated every tile of its subtile).
            // A stage is released as soon as its columns are in registers, before they are tested.
            // The no-hit path of a unit is its read-out, one min tree over its 64 columns and one vote: a warp meets a hit
            // in about one unit in twelve on the seeded d = 16 scan, so everything the search for the hit columns needs
            // (block minima, column bits, the tail-tile mask) is computed only on the units that have one.
            constexpr int G = SW / 32;          // 32-column groups per unit
            static_assert(NUM_ACC == U, "unit h of every tile uses accumulator stage h");
            uint32_t r[G][32];
            // per-warp constants: unit h reads stage h at taddr0 + h MT SW and waits on / releases barrier h MT + mt
            // (a shuffled value: ptxas keeps it instead of rebuilding it from the warp index on every unit)
            const uint32_t taddr0 = __shfl_sync(full, tmem_base + ((uint32_t)(quad * 32) << 16) + mt * SW, 0);
            uint64_t* const tfull_w = tfull_bar + mt;
            uint64_t* const tempty_w = tempty_bar + mt;
            // hit columns of one 32-column group [col0, col0 + 32) of tile j, searched in blocks of 8: a column is a
            // candidate iff its value is <= theta (never a NaN)
            auto hit_bits = [&](const uint32_t (&rg)[32], uint32_t j, int col0) -> uint32_t {
                uint32_t bits = 0;
#pragma unroll
                for (int b = 0; b < 4; ++b) {
                    const float x0 = fminf(__uint_as_float(rg[8 * b]), fminf(__uint_as_float(rg[8 * b + 1]), __uint_as_float(rg[8 * b + 2])));
                    const float x1 = fminf(__uint_as_float(rg[8 * b + 3]), fminf(__uint_as_float(rg[8 * b + 4]), __uint_as_float(rg[8 * b + 5])));
                    const float mb = fminf(fminf(x0, x1), fminf(__uint_as_float(rg[8 * b + 6]), __uint_as_float(rg[8 * b + 7])));
                    if (mb <= theta) {
#pragma unroll
                        for (int i = 0; i < 8; ++i) bits |= (__uint_as_float(rg[8 * b + i]) <= theta ? 1u : 0u) << (8 * b + i);
                    }
                }
                if (j + 1 == a.n_tiles) {  // rows past the last point are zero-filled
                    const int valid = (int)t.n - (int)(j * BN + col0);
                    if (valid < 32) bits &= valid > 0 ? ((1u << valid) - 1u) : 0u;
                }
                return bits;
            };
            PROF_DECL;
            uint32_t jn = j_begin;  // counted along: computing j_begin + jr makes ptxas rebuild j_begin from blockIdx.y every tile
            for (uint32_t jr = 0; jr < n_my; ++jr, ++jn) {
                const uint32_t j = PRUNE ? titer.next() : jn;  // absolute tile (point rows); stage and phase follow the CTA's own count
                const uint32_t aph = jr & 1u;                  // both stages complete once per tile
#pragma unroll
                for (int h = 0; h < U; ++h) {
                    PROF_ADD(3);
                    mbar_wait(tfull_w + h * MT, aph);
                    tc_fence_after();
                    PROF_ADD(0);
                    if (lane == 0 && h == 0) TRACE(warp, j, 0);
    #pragma unroll
                    for (int g = 0; g < G; ++g) tmem_ld32_issue(taddr0 + h * MT * SW + g * 32, r[g]);
                    tmem_ld_wait(r);
                    tc_fence_before();
                    __syncwarp();
                    if (elect_one()) mbar_arrive(tempty_w + h * MT);  // one lane: unlike lane == 0 it needs no thread index
                    PROF_ADD(1);
                    if (lane == 0 && h == 0) TRACE(warp, j, 1);
    #ifdef PN_TC_PROFILE
                    if (a.dbg & 1u) continue;
    #endif
                    if (__any_sync(full, unit_min64(r) <= theta)) {
                        // both groups are searched against the same theta before either is pushed
                        uint32_t bits[G];
    #pragma unroll
                        for (int g = 0; g < G; ++g) bits[g] = hit_bits(r[g], j, (h * G + g) * 32);
    #pragma unroll
                        for (int g = 0; g < G; ++g) push32(bits[g], j, (h * G + g) * 32);
                    }
                    PROF_ADD(2);
                }
                if (lane == 0) TRACE(warp, j, 2);
                // scheduled drain: every warp of the CTA drains in the same tile, so the stalls coincide
                if (((PRUNE ? jr : j) & 31u) == 31u) {
                    if (qn > 0) { drain(qn); qn = 0; __syncwarp(); }
                    if (SHARED && gb) refresh_theta(false);  // pick up the other splits' progress
                }
                if (lane == 0) TRACE(warp, j, 3);
            }
            if (warp == 0 && lane == 0) PROF_FLUSH(6);
        } else {
            constexpr int H = MT > 2 ? 2 : 1;   // read-out halves per stage
            constexpr int G = BN / 32 / H;      // 32-column groups per half
            uint32_t r[G][32];
            const uint32_t lane_off = (uint32_t)(quad * 32) << 16;
            PROF_DECL;
            for (uint32_t jr = 0; jr < n_my; ++jr) {
                const uint32_t j = PRUNE ? titer.next() : j_begin + jr;  // absolute tile (point rows); stage and phase follow the CTA's own count
                const uint32_t as = jr % NUM_ACC, aph = (jr / NUM_ACC) & 1u;
                PROF_ADD(3);
                mbar_wait(&tfull_bar[as * MT + mt], aph);
                tc_fence_after();
                PROF_ADD(0);
                if (lane == 0) TRACE(warp, j, 0);
                const uint32_t taddr = tmem_base + lane_off + (as * MT + mt) * BN;
                uint32_t bits[H * G];  // hit masks (H = 2)
                uint32_t any = 0;  // groups with a hit in some lane (warp-uniform)
    #pragma unroll
                for (int h = 0; h < H; ++h) {
    #pragma unroll
                    for (int g = 0; g < G; ++g) tmem_ld32_issue(taddr + (h * G + g) * 32, r[g]);
    #pragma unroll
                    for (int g = 0; g < G; ++g) tmem_ld_wait(r[g]);
                    if (h == H - 1) {
                        // the stage is released as soon as its last column is in registers, BEFORE that half is
                        // tested: the MMA -> read-out -> release loop of a stage is the critical path
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) mbar_arrive(&tempty_bar[as * MT + mt]);
                        PROF_ADD(1);
                        if (lane == 0) TRACE(warp, j, 1);
                    }
    #ifdef PN_TC_PROFILE
                    if (a.dbg & 1u) continue;
    #endif
                    // every test comes before any push, so that the variable-length part (queue pushes, exact reranks)
                    // never delays the next read-out
    #pragma unroll
                    for (int g = 0; g < G; ++g) any |= test32(r[g], j, (h * G + g) * 32, bits[h * G + g]) ? 1u << (h * G + g) : 0u;
                }
                if (any) {
    #pragma unroll
                    for (int g = 0; g < H * G; ++g)
                        if (any & (1u << g)) push32(bits[g], j, g * 32);
                }
                PROF_ADD(2);
                if (lane == 0) TRACE(warp, j, 2);
                // scheduled drain: every warp of the CTA drains in the same tile, so the stalls coincide
                if (((PRUNE ? jr : j) & 31u) == 31u) {
                    if (qn > 0) { drain(qn); qn = 0; __syncwarp(); }
                    if (SHARED && gb) refresh_theta(false);  // pick up the other splits' progress
                }
                if (lane == 0) TRACE(warp, j, 3);
            }
            if (warp == 0 && lane == 0) PROF_FLUSH(6);
        }
        if (qn > 0) { drain(qn); qn = 0; }
        if (active) {
            const size_t base = ((size_t)blockIdx.y * (a.nq - a.row0) + (qrow - a.row0)) * a.k;
            topk.store(a.part_d + base, a.part_i + base);
        }
        if (a.counters && lane == 0) atomicAdd(&a.counters[2], hits);
    }

    tc_fence_before();
    __syncthreads();
    if (warp == EPI_WARPS + 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
    }
}

}  // namespace tc
}  // namespace petal
