// Shared declarations of the MSM translation units (see msm.cu for the pipeline overview).
#pragma once
#include "ctx.hpp"
#include "g1.cuh"

namespace swb {

constexpr int MSM_MAX_WINDOWS = 128;
constexpr int MSM_PAIR_MAX_LEVELS = 4;   // summed blocks of up to 16 positions (the shortest accumulation range)
// sorted pairs from which batch-affine pair sums run automatically.  Measured: +9 % at 2^24 points, +12 % at 2^26, a 1/8
// bucket share of 2^26 (92 M pairs) +3-7 %; the batched and single MSMs of a 2^20-constraint prover (17-160 M pairs, 26-100
// per bucket) 0.334 -> 0.327 s with tables and 0.402 -> 0.375 s without; below 2^24 pairs the fixed cost of the block-wide
// inversions loses (2^16 constraints: 44 -> 51 ms with the threshold at 2^22)
constexpr size_t MSM_PAIR_MIN_PAIRS = (size_t)1 << 24;
// block size of the heavy-bucket gather: a bucket that holds a large share of all points (scalars equal to
// one, top window) has one partial sum per range, i.e. up to ~10^5 of them, summed by one block
constexpr int MSM_HEAVY_THREADS = 256;
constexpr int MSM_HEAVY_CHUNK = 4096;  // partial sums of a heavy bucket that one block adds up
// block size of the other bucket-tail kernels (gather, segments, bit sums): small enough (64 x <= 170
// registers) to fit beside two resident blocks of another MSM's accumulation kernel, so the tail of one
// MSM really runs under the accumulation of the next
constexpr int MSM_TAIL_THREADS = 64;
constexpr int MSM_SEG_LEN = 32;        // longest segment of the bucket reduction's running-sum level
constexpr int MSM_GATHER_INLINE = 32;  // buckets with more partial sums than this go to the block-wide path

constexpr int MSM_SEG_MIN = 4;         // shortest segment (used while there are few segments)

// Segment length of the running-sum level of the bucket reduction: every thread walks its segment
// serially (two additions per bucket, 15-25 us each for a lone thread), so short segments while there
// are too few of them to fill the GPU, MSM_SEG_LEN once there are plenty.
inline uint32_t msm_reduce_seg_len(uint32_t nwin, uint32_t B) {
    uint32_t L = B < (uint32_t)MSM_SEG_LEN ? B : (uint32_t)MSM_SEG_LEN;
    while (L > (uint32_t)MSM_SEG_MIN && (size_t)nwin * (B / L) < 32768) L >>= 1;
    return L;
}

// the sort ping-pongs between two halves of the key / value buffers; the second half starts on a
// 256-byte boundary so that the accumulation kernel can read either with 16-byte loads
inline size_t msm_alt_offset(size_t total) { return (total + 63) & ~(size_t)63; }


// the scalar vectors of a (possibly batched) MSM: vector k has start[k + 1] - start[k] scalars whose bases begin at
// record offset[k] of the handle
struct MsmBatch {
    const uint32_t* scalars[MSM_MAX_BATCH];
    uint32_t start[MSM_MAX_BATCH + 1];
    uint32_t offset[MSM_MAX_BATCH];
    uint32_t count;
};

struct MsmPlan {
    size_t n;            // points (all vectors of a batch together)
    int cb;              // window bits
    int ndig;            // digits (windows) per scalar
    int nwin;            // bucket sets: ndig on the plain path, 1 with window tables
    size_t seg_len;      // pairs per bucket set: n on the plain path, n * ndig with window tables
    size_t tab_stride;   // records per table level (0 = plain path)
    uint32_t B;          // buckets per set that this call fills: 2^(cb-1), or that divided by the bucket-shard world
    uint32_t shard_rank, shard_shift;   // bucket sharding: ours are the buckets b with b mod 2^shift == rank, stored at b >> shift
    bool idle;           // bucket shard with too few buckets to split: rank 0 computes all of it, this rank contributes the identity
    bool compact;        // table path under bucket sharding: only the pairs of our buckets are kept (total is then
                         // known after the digits kernel)
    uint32_t nb;         // total buckets = nwin * B
    uint32_t key_space;  // keys below this are buckets, the value itself marks "no bucket": B when every bucket set has its
                         // own segment of the pair list, nb for a batch (sets told apart by the key, one segment)
    size_t total;        // n * ndig (bucket, point) pairs
    uint32_t range_len;  // sorted positions per accumulation thread
    uint32_t nranges;    // ceil(total / range_len)
    uint32_t pcap;       // capacity of the partial-sum list (nranges + nb)
    int pair_levels;     // levels of batch-affine pair sums in front of the accumulation (0 = none)
};

// plans what depends on the number of sorted pairs (pl.total): the accumulation ranges and the pair-sum levels.  msm_plan
// calls it, and msm_launch_digits_sort again once a compacting digits kernel has counted the pairs it kept.
void msm_plan_pairs(const swb_ctx* c, MsmPlan& pl);

struct MsmBuffers {
    uint32_t* keys;      // [2][msm_alt_offset(total)]
    uint32_t* vals;      // [2][msm_alt_offset(total)]
    uint32_t* range_off; // [nranges + 1] runs per range, scanned in place: where each range writes
    uint32_t* pkey;      // [pcap] bucket id of each partial sum
    uint32_t* pstart;    // [nb + 1] first partial of each bucket
    uint32_t* heavy;     // [1 + nb] counter + list of buckets with many partial sums
    G1Xyzz* partial;     // [pcap]
    G1Xyzz* buckets;     // [nb]
    G1Xyzz* seg;         // [2][nwin * B / L]  per-segment weighted and plain sums of the bucket reduction
    G1Xyzz* seg2;        // per-job partial sums and values of the bucket reduction
    G1Xyzz* wins;        // [2][MSM_MAX_WINDOWS]: weighted sums sum_k (k+1) B_k, then plain sums sum_k B_k (bucket shards)
    uint32_t* count;     // [1] pairs kept by the compacting digits kernel
    Fq* pair_sums[MSM_PAIR_MAX_LEVELS + 1];    // [l]: ceil(total / 2^l) slots of two field elements (msm_pairs.cu)
    uint8_t* pair_lvl;                         // [ceil(total / 2)] level map read by k_msm_accumulate_paired
};

// msm_sort.cu: digits, sort, per-range run counts and their scan
int msm_launch_digits_sort(swb_ctx* c, MsmPlan& pl, const MsmBuffers& bf, const MsmBatch& batch, int montgomery,
                           const uint32_t** sorted_keys, const uint32_t** sorted_vals, StageTimer* tm);
// msm_accumulate.cu: one thread per range of sorted pairs -> partial sums
int msm_launch_accumulate(swb_ctx* c, const MsmPlan& pl, const MsmBuffers& bf, const uint32_t* sorted_keys,
                          const uint32_t* sorted_vals, const Fq* bases);
// msm_pairs.cu: batch-affine sums of neighbouring same-bucket positions
int msm_launch_pair_sums(swb_ctx* c, const MsmPlan& pl, Fq* const* R, uint8_t* lvl, int levels, const uint32_t* sorted_keys,
                         const uint32_t* sorted_vals, const Fq* bases, StageTimer* tm);
// msm_reduce.cu: partial sums -> buckets -> window sums
int msm_launch_gather(swb_ctx* c, const MsmPlan& pl, const MsmBuffers& bf);
int msm_launch_reduce(swb_ctx* c, const MsmPlan& pl, const MsmBuffers& bf);

}  // namespace swb
