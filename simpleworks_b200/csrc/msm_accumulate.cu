// MSM stage 4: bucket accumulation -- the dominant kernel (n * W mixed additions).
//
// Work is split by POSITION in the sorted pair list, not by bucket: thread r adds the points of
// sorted positions [r*len, (r+1)*len) and emits one XYZZ partial sum per run of equal bucket ids.
// Every lane therefore performs the same number of mixed additions whatever the digit
// distribution (a bucket holding half of all points -- top window, or scalars equal to 1 -- is
// simply spread over many threads), and a bucket that straddles ranges gets several partial sums
// which msm_reduce.cu adds up.
#include "msm_common.cuh"

namespace swb {

__device__ __forceinline__ G1Aff ld_aff(const Fq* __restrict__ xy, size_t i) {
    const uint4* q = reinterpret_cast<const uint4*>(xy + 2 * i);
    G1Aff p;
#pragma unroll
    for (int k = 0; k < 3; k++) {
        uint4 a = q[k];
        p.x.l[4 * k] = a.x; p.x.l[4 * k + 1] = a.y; p.x.l[4 * k + 2] = a.z; p.x.l[4 * k + 3] = a.w;
    }
#pragma unroll
    for (int k = 0; k < 3; k++) {
        uint4 a = q[3 + k];
        p.y.l[4 * k] = a.x; p.y.l[4 * k + 1] = a.y; p.y.l[4 * k + 2] = a.z; p.y.l[4 * k + 3] = a.w;
    }
    return p;
}


__global__ void __launch_bounds__(128) k_msm_accumulate(G1Xyzz* __restrict__ partial, uint32_t* __restrict__ pkey,
                                                         const uint32_t* __restrict__ range_off,
                                                         const uint32_t* __restrict__ keys, const uint32_t* __restrict__ vals,
                                                         const Fq* __restrict__ bases, size_t total, size_t n, uint32_t B,
                                                         uint32_t len, uint32_t nranges) {
    // The thread walks its range sequentially; reading keys/vals one word at a time would fetch a
    // whole DRAM sector per word for every lane (ranges are len*4 bytes apart).  So each thread pulls
    // 8 positions (two 16-byte loads per array) into its own column of a small shared-memory queue.
    __shared__ uint32_t qk[8][128], qv[8][128];
    const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= nranges) return;
    const uint32_t t = threadIdx.x;
    const size_t p0 = (size_t)r * len;                      // len is a power of two >= 16: 32-byte aligned chunks
    const size_t p1 = p0 + len < total ? p0 + len : total;
    auto fetch = [&](size_t q, uint32_t* k, uint32_t* v) {
        const uint32_t j = (uint32_t)(q - p0) & 7u;
        if (j == 0) {
            if (q + 8 <= total) {
                const uint4 k0 = *reinterpret_cast<const uint4*>(keys + q), k1 = *reinterpret_cast<const uint4*>(keys + q + 4);
                const uint4 v0 = *reinterpret_cast<const uint4*>(vals + q), v1 = *reinterpret_cast<const uint4*>(vals + q + 4);
                qk[0][t] = k0.x; qk[1][t] = k0.y; qk[2][t] = k0.z; qk[3][t] = k0.w;
                qk[4][t] = k1.x; qk[5][t] = k1.y; qk[6][t] = k1.z; qk[7][t] = k1.w;
                qv[0][t] = v0.x; qv[1][t] = v0.y; qv[2][t] = v0.z; qv[3][t] = v0.w;
                qv[4][t] = v1.x; qv[5][t] = v1.y; qv[6][t] = v1.z; qv[7][t] = v1.w;
            } else {
                for (uint32_t e = 0; q + e < total; e++) {
                    qk[e][t] = keys[q + e];
                    qv[e][t] = vals[q + e];
                }
            }
        }
        *k = qk[j][t];
        *v = qv[j][t];
    };
    uint32_t out = range_off[r];
    uint32_t cur = 0xffffffffu;
    G1Xyzz acc = G1Xyzz::identity();
    // bucket set of position p is p / n; tracked incrementally (a range may cross set boundaries)
    uint32_t set_base = (uint32_t)(p0 / n) * B;
    size_t set_end = (p0 / n + 1) * n;
    // software pipeline: the next point is in flight while the current one is added
    uint32_t k_next, v_next;
    fetch(p0, &k_next, &v_next);
    G1Aff pt_next;
    if (k_next < B) pt_next = ld_aff(bases, v_next & 0x7fffffffu);
    for (size_t p = p0; p < p1; p++) {
        const uint32_t kl = k_next, v = v_next;
        G1Aff pt = pt_next;
        if (p + 1 < p1) {
            fetch(p + 1, &k_next, &v_next);
            if (k_next < B) pt_next = ld_aff(bases, v_next & 0x7fffffffu);
        }
        if (p == set_end) {
            set_base += B;
            set_end += n;
        }
        if (kl >= B) continue;                              // zero digit (tail of a set's segment)
        const uint32_t k = set_base + kl;                   // global bucket id
        if (k != cur) {
            if (cur != 0xffffffffu) {
                partial[out] = acc;
                pkey[out] = cur;
                out++;
            }
            cur = k;
            acc = G1Xyzz::identity();
        }
        if (pt.is_identity()) continue;
        if (v >> 31) pt.y = pt.y.neg();
        acc.add_affine(pt.x, pt.y);
    }
    if (cur != 0xffffffffu) {
        partial[out] = acc;
        pkey[out] = cur;
    }
}

// The same walk over a range of sorted positions after msm_pairs.cu has pair-summed them: lvl[p / 2] = L > 0 says that the
// 2^L positions starting at the even position p are one bucket's points and R_L[p >> L] is their affine sum -- ONE mixed
// addition for the whole block; L = 0 leaves the two table points of (p, p + 1) to be added as in k_msm_accumulate.
struct PairLevels {
    const Fq* R[MSM_PAIR_MAX_LEVELS + 1];
    const uint8_t* lvl;
};
__global__ void __launch_bounds__(128) k_msm_accumulate_paired(G1Xyzz* __restrict__ partial, uint32_t* __restrict__ pkey,
                                                                const uint32_t* __restrict__ range_off,
                                                                const uint32_t* __restrict__ keys, const uint32_t* __restrict__ vals,
                                                                const Fq* __restrict__ bases, PairLevels pv, size_t total,
                                                                size_t n, uint32_t B, uint32_t len, uint32_t nranges) {
    const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= nranges) return;
    const size_t p0 = (size_t)r * len;                      // len is a power of two >= 16: blocks of up to 16 positions never straddle ranges
    const size_t p1 = p0 + len < total ? p0 + len : total;
    uint32_t out = range_off[r];
    uint32_t cur = 0xffffffffu;
    G1Xyzz acc = G1Xyzz::identity();
    uint32_t set_base = (uint32_t)(p0 / n) * B;
    size_t set_end = (p0 / n + 1) * n;
    // ONE point per iteration through ONE copy of the addition code, whatever its origin: lanes of a warp that are at
    // different kinds of positions do not diverge into separate copies of a 3000-instruction addition.
    size_t p = p0;                 // next position to look at (even unless `second`)
    bool second = false;           // the second table point of an unsummed pair is due
    while (p < p1) {
        while (p >= set_end) {                               // the bucket set of position p (no division in the loop)
            set_base += B;
            set_end += n;
        }
        const uint32_t kl = keys[p];
        uint32_t v = 0;
        const Fq* src;
        if (!second) {
            const uint32_t L = pv.lvl[p >> 1];
            if (L) {
                src = pv.R[L] + 2 * (p >> L);
                p += (size_t)1 << L;
            } else {
                v = vals[p];
                src = bases + 2 * (size_t)(v & 0x7fffffffu);
                second = p + 1 < p1;
                p += 1;
            }
        } else {
            v = vals[p];
            src = bases + 2 * (size_t)(v & 0x7fffffffu);
            second = false;
            p += 1;
        }
        if (kl >= B) continue;                                   // zero digit / another rank's bucket
        G1Aff pt = ld_aff(src, 0);
        const uint32_t k = set_base + kl;
        if (k != cur) {
            if (cur != 0xffffffffu) {
                partial[out] = acc;
                pkey[out] = cur;
                out++;
            }
            cur = k;
            acc = G1Xyzz::identity();
        }
        if (pt.is_identity()) continue;
        if (v >> 31) pt.y = pt.y.neg();
        acc.add_affine(pt.x, pt.y);
    }
    if (cur != 0xffffffffu) {
        partial[out] = acc;
        pkey[out] = cur;
    }
}

int msm_launch_accumulate(swb_ctx* c, const MsmPlan& pl, const MsmBuffers& bf, const uint32_t* sorted_keys,
                          const uint32_t* sorted_vals, const Fq* bases) {
    if (pl.nranges == 0) return SWB_OK;      // a bucket shard that received no pairs
    if (pl.pair_levels > 0) {
        PairLevels pv{};
        for (int l = 1; l <= pl.pair_levels; l++) pv.R[l] = bf.pair_sums[l];
        pv.lvl = bf.pair_lvl;
        k_msm_accumulate_paired<<<(pl.nranges + 127) / 128, 128, 0, c->stream>>>(bf.partial, bf.pkey, bf.range_off, sorted_keys,
                                                                                sorted_vals, bases, pv, pl.total, pl.seg_len,
                                                                                pl.key_space, pl.range_len, pl.nranges);
        SWB_LAUNCH_CHECK(c, "k_msm_accumulate_paired");
        return SWB_OK;
    }
    k_msm_accumulate<<<(pl.nranges + 127) / 128, 128, 0, c->stream>>>(bf.partial, bf.pkey, bf.range_off, sorted_keys, sorted_vals,
                                                                     bases, pl.total, pl.seg_len, pl.key_space, pl.range_len, pl.nranges);
    SWB_LAUNCH_CHECK(c, "k_msm_accumulate");
    return SWB_OK;
}

}  // namespace swb
