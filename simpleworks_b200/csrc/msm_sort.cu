// MSM stages 1-3: signed-digit decomposition, radix sort of (bucket, point) pairs (radix_sort.cu),
// and the per-range run counts that tell the accumulation kernel where to write.
#include "msm_common.cuh"
#include "radix_sort.hpp"

namespace swb {

// ---- 1. signed-digit decomposition --------------------------------------------------------
__device__ __forceinline__ bool fr_geq_mod(const uint32_t* a) {   // a (8 limbs) >= r
    for (int k = 7; k >= 0; k--) {
        const uint32_t m = FrParams::mod(k);
        if (a[k] != m) return a[k] > m;
    }
    return true;
}
__device__ __forceinline__ void fr_sub_mod(uint32_t* a) {         // a -= r
    uint64_t borrow = 0;
    for (int k = 0; k < 8; k++) {
        const uint64_t d = (uint64_t)a[k] - FrParams::mod(k) - borrow;
        a[k] = (uint32_t)d;
        borrow = (d >> 32) & 1u;
    }
}
__device__ __forceinline__ void fr_mod_minus(uint32_t* a) {       // a = r - a
    uint64_t borrow = 0;
    for (int k = 0; k < 8; k++) {
        const uint64_t d = (uint64_t)FrParams::mod(k) - a[k] - borrow;
        a[k] = (uint32_t)d;
        borrow = (d >> 32) & 1u;
    }
}

// scalar i of the batch: canonical limbs (on the table path reduced to <= r/2, flip = 1 if it was negated), the first key of
// its bucket set and its base record; false past the end
__device__ __forceinline__ bool digits_load(const MsmBatch& batch, size_t i, size_t n, int montgomery, size_t tab_stride,
                                            uint32_t Bloc, Fr& s, uint32_t& flip, uint32_t& key0, size_t& rec) {
    s = Fr::zero();
    flip = 0;
    key0 = 0;
    rec = 0;
    if (i >= n) return false;
    uint32_t vec = 0;                                   // which vector of the batch scalar i belongs to
    while (vec + 1 < batch.count && (uint32_t)i >= batch.start[vec + 1]) vec++;
    key0 = vec * Bloc;
    rec = (size_t)batch.offset[vec] + (i - batch.start[vec]);
    const uint4* q = reinterpret_cast<const uint4*>(batch.scalars[vec] + 8 * (i - batch.start[vec]));
    uint4 a = q[0], b = q[1];
    s.l[0] = a.x; s.l[1] = a.y; s.l[2] = a.z; s.l[3] = a.w;
    s.l[4] = b.x; s.l[5] = b.y; s.l[6] = b.z; s.l[7] = b.w;
    if (montgomery) s = s.to_canonical();
    if (tab_stride) {
        if ((s.l[7] >> 28) != 0)                              // r < 2^253 < 2^28 * 2^224: anything below is canonical
            while (fr_geq_mod(s.l)) fr_sub_mod(s.l);          // non-canonical input: reduce first
        uint32_t t[8];                                    // 2s >= r  <=>  s > r/2
        uint32_t top = 0;
        for (int k = 0; k < 8; k++) {
            t[k] = (s.l[k] << 1) | top;
            top = s.l[k] >> 31;
        }
        if (top || fr_geq_mod(t)) {
            fr_mod_minus(s.l);
            flip = 1;
        }
    }
    return true;
}

// Plain path (tab_stride == 0): window w of scalar i -> keys[w*n + i] = |d| - 1 (or B when d == 0:
// sorts to the end of the window's segment), vals[w*n + i] = i | sign << 31; nwin covers 254 bits so
// that the top carry has a window of its own, and nothing is assumed about the bases.
// Table path (tab_stride == N > 0): the point of window w is table entry w*N + i, all windows share
// the buckets, and a scalar above r/2 is replaced by r - s with every sign flipped (bases in the
// prime-order subgroup), so nwin = ceil(253 / c) windows suffice.
// Bucket sharding (shift > 0): only the digits whose bucket b has b mod 2^shift == rank are ours (interleaved, so
// that every rank gets the same load whatever the digit distribution -- the top window of a 253-bit scalar only
// reaches the lower buckets); keys are local (b >> shift) and every other digit gets the marker Bloc, like a
// zero digit.  With COMPACT
// (table path: one bucket set, so the order of the pairs is free) the marked pairs are not written at
// all: a block counts what it keeps in shared memory, reserves the space with one atomicAdd on *count and
// writes its pairs there -- the arrays the sort sees shrink with the number of ranks.
// A batch (several scalar vectors over one bases handle, table path only) gives vector k its own bucket set: its keys are
// k * Bloc + bucket, its points start at record batch.offset[k]; the marker is the number of buckets of the whole batch.
// The window width C is a template parameter, so every window position is a constant: a digit costs two shifts, and the
// digits and warp votes of all windows stay in registers, so nothing is computed twice (ncu, 2^26 scalars, 1/8 bucket
// share: with the width known only at run time, the scalar walked through a 256-bit shift register, the kernel executed
// ~950 warp instructions per 32 scalars and was issue-bound at 2.4-2.6 ms; with it fixed, 1.9 ms).  Measured and dropped:
// splitting the compaction into two barrier-free kernels (count per warp, scan, place) -- 420 + 665 instructions per 32
// scalars, 2.7 ms.
template <int C>
struct Digits {
    static constexpr int NW = (254 + C - 1) / C;          // nwin <= NW
    static constexpr uint32_t CM = (1u << C) - 1u, B = 1u << (C - 1);
    // |digit| with the sign (already combined with `flip`) in bit 31; 0: nothing to add
    static __device__ __forceinline__ void digits(const Fr& s, bool live, uint32_t flip, int nwin, uint32_t (&d)[NW]) {
        uint32_t carry = 0;
#pragma unroll
        for (int w = 0; w < NW; w++) {
            const int bit = w * C, limb = bit >> 5, off = bit & 31;
            uint32_t v = 0;
            if (limb < 8) {
                v = s.l[limb] >> off;
                if (off + C > 32 && limb + 1 < 8) v |= s.l[limb + 1] << (32 - off);
            }
            v = (v & CM) + carry;
            const uint32_t neg = v > B ? 1u : 0u;
            if (neg) v = (1u << C) - v;
            carry = neg;
            d[w] = (live && w < nwin && v) ? (v | ((neg ^ flip) << 31)) : 0u;
        }
    }
};

template <bool COMPACT, int C>
__global__ void __launch_bounds__(256) k_msm_digits(uint32_t* __restrict__ keys, uint32_t* __restrict__ vals,
                                                     MsmBatch batch, size_t n, int nwin,
                                                     int montgomery, size_t tab_stride, uint32_t rank, uint32_t shift, uint32_t Bloc,
                                                     uint32_t* __restrict__ count) {
    using D = Digits<C>;
    const uint32_t marker = Bloc * batch.count;
    const uint32_t smask = (1u << shift) - 1u;
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    __shared__ uint32_t s_cnt, s_base;
    const size_t rounds = (n + stride - 1) / stride;      // compaction is block-wide: every thread runs every round
    for (size_t round = 0; round < rounds; round++, i += stride) {
        Fr s;
        uint32_t flip, key0;
        size_t rec;
        const bool live = digits_load(batch, i, n, montgomery, tab_stride, Bloc, s, flip, key0, rec);
        uint32_t d[D::NW];
        D::digits(s, live, flip, nwin, d);
        if (!COMPACT) {
            if (live) {
#pragma unroll
                for (int w = 0; w < D::NW; w++) {
                    if (w < nwin) {
                        const uint32_t v = d[w] & 0x7fffffffu;
                        const uint32_t key = (v && ((v - 1) & smask) == rank) ? key0 + ((v - 1) >> shift) : marker;
                        keys[(size_t)w * n + i] = key;
                        vals[(size_t)w * n + i] = (uint32_t)(tab_stride ? (size_t)w * tab_stride + rec : rec) | (d[w] & 0x80000000u);
                    }
                }
            }
            continue;
        }
        // count, reserve (one global atomic per block and round), write; a warp's pairs are laid out window by window,
        // so that the lanes keeping window w write neighbouring slots
        if (threadIdx.x == 0) s_cnt = 0;
        __syncthreads();
        const uint32_t lane = threadIdx.x & 31u;
        uint32_t who[D::NW], warp_total = 0;
#pragma unroll
        for (int w = 0; w < D::NW; w++) {
            const uint32_t v = d[w] & 0x7fffffffu;
            who[w] = __ballot_sync(0xffffffffu, v && ((v - 1) & smask) == rank);
            warp_total += (uint32_t)__popc(who[w]);
        }
        uint32_t warp_base = 0;
        if (lane == 0 && warp_total) warp_base = atomicAdd(&s_cnt, warp_total);
        warp_base = __shfl_sync(0xffffffffu, warp_base, 0);
        __syncthreads();
        if (threadIdx.x == 0) s_base = s_cnt ? atomicAdd(count, s_cnt) : 0u;
        __syncthreads();
        uint32_t seg = s_base + warp_base;
        const uint32_t below = (1u << lane) - 1u;
#pragma unroll
        for (int w = 0; w < D::NW; w++) {
            if ((who[w] >> lane) & 1u) {
                const uint32_t at = seg + (uint32_t)__popc(who[w] & below);
                keys[at] = key0 + (((d[w] & 0x7fffffffu) - 1) >> shift);
                vals[at] = (uint32_t)((size_t)w * tab_stride + rec) | (d[w] & 0x80000000u);
            }
            seg += (uint32_t)__popc(who[w]);
        }
    }
}

// launches k_msm_digits<pl.compact, pl.cb>.  Every width the plan can choose has one: c in [2, 24] on the plain path
// (swb_msm_set_window_bits, pick_window), c in [8, 24] over tables (swb_bases_precompute), and only tables compact.
template <int C>
static int msm_launch_digits(swb_ctx* c, const MsmPlan& pl, const MsmBuffers& bf, const MsmBatch& batch, int montgomery,
                             unsigned blocks) {
    if (pl.ndig > Digits<C>::NW) return set_err(c, SWB_EINTERNAL, "msm: %d digits of %d bits exceed the digits kernel", pl.ndig, C);
    if (!pl.compact)
        k_msm_digits<false, C><<<blocks, 256, 0, c->stream>>>(bf.keys, bf.vals, batch, pl.n, pl.ndig, montgomery, pl.tab_stride,
                                                               pl.shard_rank, pl.shard_shift, pl.B, nullptr);
    else if constexpr (C >= 8)
        k_msm_digits<true, C><<<blocks, 256, 0, c->stream>>>(bf.keys, bf.vals, batch, pl.n, pl.ndig, montgomery, pl.tab_stride,
                                                              pl.shard_rank, pl.shard_shift, pl.B, bf.count);
    else
        return set_err(c, SWB_EINTERNAL, "msm: no compacting digits kernel for c = %d (window tables have c >= 8)", C);
    SWB_LAUNCH_CHECK(c, "k_msm_digits");
    return SWB_OK;
}

static int msm_launch_digits(swb_ctx* c, const MsmPlan& pl, const MsmBuffers& bf, const MsmBatch& batch, int montgomery,
                             unsigned blocks) {
    switch (pl.cb) {
#define SWB_DIGITS_CASE(CB) \
    case CB: return msm_launch_digits<CB>(c, pl, bf, batch, montgomery, blocks);
        SWB_DIGITS_CASE(2) SWB_DIGITS_CASE(3) SWB_DIGITS_CASE(4) SWB_DIGITS_CASE(5) SWB_DIGITS_CASE(6) SWB_DIGITS_CASE(7)
        SWB_DIGITS_CASE(8) SWB_DIGITS_CASE(9) SWB_DIGITS_CASE(10) SWB_DIGITS_CASE(11) SWB_DIGITS_CASE(12) SWB_DIGITS_CASE(13)
        SWB_DIGITS_CASE(14) SWB_DIGITS_CASE(15) SWB_DIGITS_CASE(16) SWB_DIGITS_CASE(17) SWB_DIGITS_CASE(18) SWB_DIGITS_CASE(19)
        SWB_DIGITS_CASE(20) SWB_DIGITS_CASE(21) SWB_DIGITS_CASE(22) SWB_DIGITS_CASE(23) SWB_DIGITS_CASE(24)
#undef SWB_DIGITS_CASE
        default: return set_err(c, SWB_EINTERNAL, "msm: no digits kernel for c = %d", pl.cb);
    }
}

// ---- 3. number of runs of equal (valid) keys inside each range of `len` sorted positions -----
// Range r owns sorted positions [r*len, (r+1)*len), len a power of two >= 16.  Position p belongs
// to window p / n; its global bucket id is (p / n) * B + key, and key == B marks a zero digit (the
// tail of every window's segment).  A run is a maximal stretch of one global bucket id inside the
// range; k_msm_accumulate emits exactly one partial sum per run, so the exclusive scan of these
// counts is where each range writes.  One thread per position (coalesced), one atomic per half warp.
__global__ void __launch_bounds__(256) k_msm_range_count(uint32_t* __restrict__ cnt, const uint32_t* __restrict__ keys,
                                                          size_t total, size_t n, uint32_t B, uint32_t len) {
    const size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    bool starts = false;
    if (p < total) {
        const uint32_t k = keys[p];
        if (k < B) {
            starts = true;                                     // first position of a range or window, or after a zero digit
            if (p % len != 0 && p % n != 0) starts = keys[p - 1] != k;
        }
    }
    const uint32_t ballot = __ballot_sync(0xffffffffu, starts);
    const uint32_t lane = threadIdx.x & 31;
    if ((lane & 15) == 0 && p < total) {
        const uint32_t c = __popc(ballot & (lane ? 0xffff0000u : 0x0000ffffu));
        if (c) atomicAdd(&cnt[p / len], c);
    }
}

int msm_launch_digits_sort(swb_ctx* c, MsmPlan& pl, const MsmBuffers& bf, const MsmBatch& batch, int montgomery,
                           const uint32_t** sorted_keys, const uint32_t** sorted_vals, StageTimer* tm) {
    {
        size_t blocks = (pl.n + 255) / 256;
        size_t cap = (size_t)c->sm_count * 8;
        if (blocks > cap) blocks = cap;
        if (pl.compact) SWB_CUDA(c, cudaMemsetAsync(bf.count, 0, sizeof(uint32_t), c->stream));
        int rc = msm_launch_digits(c, pl, bf, batch, montgomery, (unsigned)blocks);
        if (rc != SWB_OK) return rc;
        if (pl.compact) {
            // the number of pairs that fell into our buckets sizes everything downstream
            uint32_t kept = 0;
            SWB_CUDA(c, cudaMemcpyAsync(&kept, bf.count, sizeof kept, cudaMemcpyDeviceToHost, c->stream));
            SWB_CUDA(c, cudaStreamSynchronize(c->stream));
            pl.total = kept;
            pl.seg_len = kept;
            msm_plan_pairs(c, pl);
        }
    }
    if (tm) tm->mark("digits");
    const size_t total = pl.total;
    if (total == 0) {                 // nothing in our bucket range: no partial sums at all
        SWB_CUDA(c, cudaMemsetAsync(bf.range_off, 0, 2 * sizeof(uint32_t), c->stream));
        *sorted_keys = bf.keys;
        *sorted_vals = bf.vals;
        return SWB_OK;
    }
    uint32_t *sk = nullptr, *sv = nullptr;
    // keys are 0 .. B (B = 2^(cb-1) marks a zero digit): cb bits, sorted inside each bucket set's segment
    int key_bits = 1;
    while ((1u << key_bits) <= pl.key_space) key_bits++;   // values 0 .. key_space
    const size_t alt = msm_alt_offset(pl.n * (size_t)pl.ndig);   // where the second halves of the buffers start
    // segments of the pair list: one per bucket set on the plain path, a single one over window tables (where a batch tells its
    // sets apart by the key)
    const uint32_t nseg = pl.tab_stride ? 1u : (uint32_t)pl.nwin;
    int rc = radix_sort_segmented(c, bf.keys, bf.keys + alt, bf.vals, bf.vals + alt, pl.seg_len, nseg, key_bits, &sk, &sv);
    if (rc != SWB_OK) return rc;
    if (tm) tm->mark("sort");
    SWB_CUDA(c, cudaMemsetAsync(bf.range_off, 0, ((size_t)pl.nranges + 1) * sizeof(uint32_t), c->stream));
    k_msm_range_count<<<(unsigned)((total + 255) / 256), 256, 0, c->stream>>>(bf.range_off, sk, total, pl.seg_len, pl.key_space, pl.range_len);
    SWB_LAUNCH_CHECK(c, "k_msm_range_count");
    rc = exclusive_scan_u32(c, bf.range_off, (size_t)pl.nranges + 1);
    if (rc != SWB_OK) return rc;
    *sorted_keys = sk;
    *sorted_vals = sv;
    return SWB_OK;
}

}  // namespace swb
