// Fixed-base powers: out[i] = beta^i * g, i < n, as affine points.
//
// Replaces what KZG10::setup does for powers_of_g / powers_of_gamma_g (ark-poly-commit 0.3
// kzg10/mod.rs): FixedBaseMSM::get_window_table + FixedBaseMSM::multi_scalar_mul over the
// powers of beta, then ProjectiveCurve::batch_normalization_into_affine.  Reached from
// Marlin::universal_setup <- reference src/marlin/mod.rs:52, simple_merkle_tree.rs:39 (1 572 862
// points per table for the (100000, 25000, 300000) bound every non-toy example uses).
//
// Device schedule: a 22 x 4096 table of d * 2^(12 o) * g (12-bit windows, affine), then one thread
// per group of 8 consecutive powers: 22 mixed additions each, one shared inversion to affine.
// Affine results are unique, so they equal arkworks' bit for bit.
#define SWB_FP_NOINLINE_MUL
#include "ctx.hpp"
#include "g1.cuh"

namespace swb {

constexpr int FB_WINDOW = 12;                         // 22 windows x 4096 entries: 8.6 MB of table, L2-resident
constexpr int FB_OUTER = (253 + FB_WINDOW - 1) / FB_WINDOW;
constexpr int FB_ENTRIES = 1 << FB_WINDOW;

__device__ __forceinline__ G1Aff xyzz_to_affine(const G1Xyzz& p) {
    G1Aff a;
    if (p.is_identity()) {
        a.x = Fq::zero();
        a.y = Fq::zero();
        return a;
    }
    Fq inv = (p.zz * p.zzz).inverse_bingcd();
    a.x = p.x * (p.zzz * inv);
    a.y = p.y * (p.zz * inv);
    return a;
}

// table[o*4096 + d] = d * 2^(12 o) * g from pow2[k] = 2^k * g
__global__ void __launch_bounds__(128) k_fb_table(G1Aff* __restrict__ table, const G1Aff* __restrict__ pow2) {
    const uint32_t e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= FB_OUTER * FB_ENTRIES) return;
    const uint32_t o = e >> FB_WINDOW, d = e & (FB_ENTRIES - 1u);
    G1Xyzz acc = G1Xyzz::identity();
    for (int b = 0; b < FB_WINDOW; b++) {
        if ((d >> b) & 1u) {
            G1Aff p = pow2[o * FB_WINDOW + b];
            if (!p.is_identity()) acc.add_affine(p.x, p.y);
        }
    }
    table[e] = xyzz_to_affine(acc);
}

// RECORD = 104: ABI GroupAffine records (x | y | infinity flag); RECORD = 96: resident base layout.
// A thread produces `group` consecutive powers (beta^(i+1) = beta^i * beta) and normalises them with
// ONE inversion (Montgomery's trick over zz * zzz, binary-GCD inversion): an inversion costs about as much as the
// 22 mixed additions of a power, so sharing it nearly halves the work.
constexpr int FB_GROUP = 8;
template <int RECORD>
__global__ void __launch_bounds__(128) k_fb_powers(uint8_t* __restrict__ out, const G1Aff* __restrict__ table, Fr beta, size_t n,
                                                    int group) {
    const size_t i0 = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) * (size_t)group;
    if (i0 >= n) return;
    const int cnt = i0 + group <= n ? group : (int)(n - i0);
    Fr bp = beta.pow_u64((uint64_t)i0);
    Fq zz[FB_GROUP], zzz[FB_GROUP], pre[FB_GROUP];
    Fq run = Fq::one();
    for (int g = 0; g < cnt; g++) {
        const Fr s = bp.to_canonical();
        bp = bp * beta;
        G1Xyzz acc = G1Xyzz::identity();
        for (int o = 0; o < FB_OUTER; o++) {
            const int bit = o * FB_WINDOW, limb = bit >> 5, off = bit & 31;
            uint32_t d = s.l[limb] >> off;
            if (off + FB_WINDOW > 32 && limb + 1 < 8) d |= s.l[limb + 1] << (32 - off);
            d &= FB_ENTRIES - 1u;
            if (d) {
                G1Aff p = table[o * FB_ENTRIES + d];
                if (!p.is_identity()) acc.add_affine(p.x, p.y);
            }
        }
        const bool inf = acc.is_identity();
        uint32_t* dst = reinterpret_cast<uint32_t*>(out + (i0 + g) * RECORD);      // X | Y for now
#pragma unroll
        for (int k = 0; k < 12; k++) dst[k] = inf ? 0u : acc.x.l[k];
#pragma unroll
        for (int k = 0; k < 12; k++) dst[12 + k] = inf ? 0u : acc.y.l[k];
        if (RECORD == 104) {
            dst[24] = inf ? 1u : 0u;
            dst[25] = 0u;
        }
        zz[g] = inf ? Fq::one() : acc.zz;
        zzz[g] = inf ? Fq::one() : acc.zzz;
        pre[g] = run;
        run = run * (zz[g] * zzz[g]);
    }
    Fq inv = run.inverse_bingcd();
    for (int g = cnt; g-- > 0;) {
        const Fq tinv = inv * pre[g];            // (zz_g * zzz_g)^-1
        inv = inv * (zz[g] * zzz[g]);
        uint32_t* dst = reinterpret_cast<uint32_t*>(out + (i0 + g) * RECORD);
        Fq x, y;
#pragma unroll
        for (int k = 0; k < 12; k++) { x.l[k] = dst[k]; y.l[k] = dst[12 + k]; }
        x = x * (tinv * zzz[g]);                 // x = X / zz
        y = y * (tinv * zz[g]);                  // y = Y / zzz
#pragma unroll
        for (int k = 0; k < 12; k++) { dst[k] = x.l[k]; dst[12 + k] = y.l[k]; }
    }
}
// enough threads to fill the GPU first, then groups that share an inversion
static inline int fb_group(size_t n) { return n >= ((size_t)1 << 18) ? FB_GROUP : 1; }

// resident 96-byte records -> 104-byte ABI records
__global__ void k_bases_export(uint8_t* __restrict__ out, const Fq* __restrict__ xy, size_t n) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t* src = reinterpret_cast<const uint32_t*>(xy + 2 * i);
    uint32_t* dst = reinterpret_cast<uint32_t*>(out + i * 104);
    uint32_t any = 0;
#pragma unroll
    for (int k = 0; k < 24; k++) { dst[k] = src[k]; any |= src[k]; }
    dst[24] = any ? 0u : 1u;
    dst[25] = 0u;
}

// ---- window tables for the MSM -------------------------------------------------------------------
// tab[j*N + i] = 2^(c*j) * base_i for j < W (level 0 = the bases themselves), all affine.  With them
// every c-bit digit of a scalar selects its own precomputed point and all W windows share ONE set of
// buckets, so the MSM needs a single bucket reduction and no Horner doublings (msm.cu).  One thread
// per base: c doublings per level in XYZZ, then one inversion for the base's W - 1 new points
// (Montgomery's trick over zz*zzz).
constexpr int TAB_MAX_LEVELS = 32;
static_assert((253 + 8 - 1) / 8 <= TAB_MAX_LEVELS, "swb_bases_precompute accepts window widths from 8 bits on");
__global__ void __launch_bounds__(128) k_bases_tables(Fq* __restrict__ tab, size_t N, int c, int W) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    G1Xyzz q = G1Xyzz::identity();
    {
        const Fq x = tab[2 * i], y = tab[2 * i + 1];
        if (!(x.is_zero() && y.is_zero())) {
            q.x = x; q.y = y;
            q.zz = Fq::one(); q.zzz = Fq::one();
        }
    }
    Fq pref[TAB_MAX_LEVELS], zz[TAB_MAX_LEVELS], zzz[TAB_MAX_LEVELS];
    Fq run = Fq::one();
    for (int j = 1; j < W; j++) {
        for (int k = 0; k < c; k++) q = q.dbl();
        const bool inf = q.is_identity();       // only for bases outside the odd-order subgroup
        tab[2 * (j * N + i)] = inf ? Fq::zero() : q.x;
        tab[2 * (j * N + i) + 1] = inf ? Fq::zero() : q.y;
        zz[j] = inf ? Fq::one() : q.zz;
        zzz[j] = inf ? Fq::one() : q.zzz;
        pref[j] = run;
        run = run * (zz[j] * zzz[j]);
    }
    Fq inv = run.inverse();
    for (int j = W - 1; j >= 1; j--) {
        const Fq tinv = inv * pref[j];          // (zz_j * zzz_j)^-1
        inv = inv * (zz[j] * zzz[j]);
        Fq* slot = tab + 2 * (j * N + i);
        slot[0] = slot[0] * (tinv * zzz[j]);    // x = X / zz
        slot[1] = slot[1] * (tinv * zz[j]);     // y = Y / zzz
    }
}

}  // namespace swb

using namespace swb;

// builds the window table for g on the device; returns it in *table
static int fb_prepare(swb_ctx* c, const swb_g1_jacobian* g_host, const swb_fr* beta_host, G1Aff** table, Fr* beta) {
    SWB_CUDA(c, cudaSetDevice(c->device));
    // host: 2^k * g for k < FB_OUTER * FB_WINDOW, affine
    G1Xyzz p;
    Fq z;
    memcpy(p.x.l, g_host->x.l, 48);
    memcpy(p.y.l, g_host->y.l, 48);
    memcpy(z.l, g_host->z.l, 48);
    if (z.is_zero()) p = G1Xyzz::identity();
    else {
        p.zz = z.sqr();
        p.zzz = p.zz * z;
    }
    // 2^k * g for every bit position, normalised with ONE inversion (Montgomery's trick; a host inversion per
    // point was 15-25 ms of every setup)
    std::vector<G1Aff> pow2(FB_OUTER * FB_WINDOW);
    {
        std::vector<G1Xyzz> pts(pow2.size());
        std::vector<Fq> pre(pow2.size());
        Fq run = Fq::one();
        for (size_t k = 0; k < pts.size(); k++) {
            pts[k] = p;
            pre[k] = run;
            if (!p.is_identity()) run = run * (p.zz * p.zzz);
            p = p.dbl();
        }
        Fq inv = run.inverse_bingcd();
        for (size_t k = pts.size(); k-- > 0;) {
            if (pts[k].is_identity()) {
                pow2[k].x = Fq::zero();
                pow2[k].y = Fq::zero();
                continue;
            }
            const Fq tinv = inv * pre[k];                  // (zz_k * zzz_k)^-1
            inv = inv * (pts[k].zz * pts[k].zzz);
            pow2[k].x = pts[k].x * (pts[k].zzz * tinv);
            pow2[k].y = pts[k].y * (pts[k].zz * tinv);
        }
    }
    memcpy(beta->l, beta_host->l, 32);
    G1Aff* d_pow2 = (G1Aff*)get_scratch(c, "fb_pow2", sizeof(G1Aff) * pow2.size());
    G1Aff* d_table = (G1Aff*)get_scratch(c, "fb_table", sizeof(G1Aff) * FB_OUTER * FB_ENTRIES);
    if (!d_pow2 || !d_table) return SWB_ENOMEM;
    SWB_CUDA(c, cudaMemcpyAsync(d_pow2, pow2.data(), sizeof(G1Aff) * pow2.size(), cudaMemcpyHostToDevice, c->stream));
    SWB_CUDA(c, cudaStreamSynchronize(c->stream));   // pow2 is a local
    k_fb_table<<<FB_OUTER * FB_ENTRIES / 128, 128, 0, c->stream>>>(d_table, d_pow2);
    SWB_LAUNCH_CHECK(c, "k_fb_table");
    *table = d_table;
    return SWB_OK;
}

extern "C" int swb_fixed_base_powers(swb_ctx* c, const swb_g1_jacobian* g_host, const swb_fr* beta_host, size_t n,
                                     swb_g1_affine* out_host) {
    if (!c) return SWB_EARG;
    SWB_REQUIRE(c, g_host && beta_host && (n == 0 || out_host), "fixed_base_powers: NULL argument");
    if (n == 0) return SWB_OK;
    G1Aff* d_table = nullptr;
    Fr beta;
    int rc = fb_prepare(c, g_host, beta_host, &d_table, &beta);
    if (rc != SWB_OK) return rc;
    uint8_t* d_out = (uint8_t*)get_scratch(c, "fb_out", n * 104);
    if (!d_out) return SWB_ENOMEM;
    {
        const int grp = fb_group(n);
        const size_t threads = (n + grp - 1) / grp;
        k_fb_powers<104><<<(unsigned)((threads + 127) / 128), 128, 0, c->stream>>>(d_out, d_table, beta, n, grp);
    }
    SWB_LAUNCH_CHECK(c, "k_fb_powers");
    SWB_CUDA(c, cudaMemcpyAsync(out_host, d_out, n * 104, cudaMemcpyDeviceToHost, c->stream));
    SWB_CUDA(c, cudaStreamSynchronize(c->stream));
    return SWB_OK;
}

extern "C" int swb_bases_from_powers(swb_ctx* c, const swb_g1_jacobian* g_host, const swb_fr* beta_host, size_t n,
                                     swb_bases** out) {
    if (!c) return SWB_EARG;
    SWB_REQUIRE(c, g_host && beta_host && out, "bases_from_powers: NULL argument");
    G1Aff* d_table = nullptr;
    Fr beta;
    int rc = fb_prepare(c, g_host, beta_host, &d_table, &beta);
    if (rc != SWB_OK) return rc;
    swb_bases* b = new swb_bases();
    b->ctx = c;
    b->n = n;
    cudaError_t e = cudaMalloc(&b->xy, (n ? n : 1) * 96);
    if (e != cudaSuccess) {
        delete b;
        return set_err(c, SWB_ENOMEM, "bases_from_powers: cudaMalloc(%zu) failed: %s", n * 96, cudaGetErrorString(e));
    }
    if (n) {
        const int grp = fb_group(n);
        const size_t threads = (n + grp - 1) / grp;
        k_fb_powers<96><<<(unsigned)((threads + 127) / 128), 128, 0, c->stream>>>((uint8_t*)b->xy, d_table, beta, n, grp);
        c->launches++;
        e = cudaGetLastError();
        if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
        if (e != cudaSuccess) {
            cudaFree(b->xy);
            delete b;
            return cuda_fail(c, e, "k_fb_powers");
        }
    }
    *out = b;
    return SWB_OK;
}

extern "C" int swb_bases_export(swb_ctx* c, const swb_bases* b, size_t offset, size_t n, swb_g1_affine* out_host) {
    if (!c) return SWB_EARG;
    SWB_REQUIRE(c, b && (n == 0 || out_host), "bases_export: NULL argument");
    SWB_REQUIRE(c, offset <= b->n && n <= b->n - offset, "bases_export: range exceeds the loaded bases");
    if (n == 0) return SWB_OK;
    SWB_CUDA(c, cudaSetDevice(c->device));
    uint8_t* d_out = (uint8_t*)get_scratch(c, "fb_out", n * 104);
    if (!d_out) return SWB_ENOMEM;
    k_bases_export<<<(unsigned)((n + 255) / 256), 256, 0, c->stream>>>(d_out, b->xy + 2 * offset, n);
    SWB_LAUNCH_CHECK(c, "k_bases_export");
    SWB_CUDA(c, cudaMemcpyAsync(out_host, d_out, n * 104, cudaMemcpyDeviceToHost, c->stream));
    SWB_CUDA(c, cudaStreamSynchronize(c->stream));
    return SWB_OK;
}

// the digit width that minimises (additions) + (bucket work) for MSMs of N scalars over window tables; the
// two weights are the measured cost of one mixed addition and of one bucket in gather + reduce
int swb::tables_pick_window(size_t N) {
    int best = 8;
    double best_cost = 1e300;
    for (int cb = 8; cb <= 23; cb++) {
        const int W = (253 + cb - 1) / cb;
        const double cost = (double)N * W * 0.37 + (double)((size_t)1 << (cb - 1)) * 3.7;
        if (cost < best_cost) { best_cost = cost; best = cb; }
    }
    return best;
}

extern "C" int swb_bases_precompute(swb_ctx* c, swb_bases* b, int window_bits) {
    if (!c) return SWB_EARG;
    SWB_REQUIRE(c, b != nullptr, "bases_precompute: NULL bases");
    SWB_REQUIRE(c, b->ctx == c, "bases_precompute: bases belong to another context");
    SWB_REQUIRE(c, window_bits == 0 || (window_bits >= 8 && window_bits <= 24), "bases_precompute: window_bits must be 0 or in [8,24]");
    if (b->tab_w) return SWB_OK;                 // already built
    if (b->n == 0) return SWB_OK;
    const int cb = window_bits ? window_bits : tables_pick_window(b->n);
    const int W = (253 + cb - 1) / cb;
    SWB_REQUIRE(c, b->n * (size_t)W < ((size_t)1 << 31), "bases_precompute: n * levels must be < 2^31");
    SWB_CUDA(c, cudaSetDevice(c->device));
    Fq* tab = nullptr;
    const size_t bytes = b->n * (size_t)W * 96;
    cudaError_t e = cudaMalloc(&tab, bytes);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return set_err(c, SWB_ENOMEM, "bases_precompute: cudaMalloc(%zu) failed: %s", bytes, cudaGetErrorString(e));
    }
    e = cudaMemcpyAsync(tab, b->xy, b->n * 96, cudaMemcpyDeviceToDevice, c->stream);
    if (e == cudaSuccess) {
        k_bases_tables<<<(unsigned)((b->n + 127) / 128), 128, 0, c->stream>>>(tab, b->n, cb, W);
        c->launches++;
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    if (e != cudaSuccess) {
        cudaFree(tab);
        return cuda_fail(c, e, "k_bases_tables");
    }
    sync_all_streams(c);                         // an MSM on a slot stream may still be reading the old records
    cudaFree(b->xy);
    b->xy = tab;
    b->tab_c = cb;
    b->tab_w = W;
    return SWB_OK;
}

extern "C" int swb_bases_table_info(const swb_bases* b, int* window_bits, int* levels) {
    if (!b) return SWB_EARG;
    if (window_bits) *window_bits = b->tab_c;
    if (levels) *levels = b->tab_w;
    return SWB_OK;
}
