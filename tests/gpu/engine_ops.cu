// Test-only shim: the prover's internal device launchers (polyops.hpp, marlin_ops.hpp) and the host
// engine's versions of the same operations (marlin/poly.hpp, marlin/rng.hpp) behind plain extern "C"
// functions, so that tests/test_gpu_engine_ops.py can call them one at a time through ctypes.
//
// Every device wrapper takes host arrays of Montgomery limbs, uploads them, runs the launcher on the
// shim's own context, synchronises and downloads the result.  Output buffers are filled with 0xFF bytes
// before the launch, so a slot the kernel never writes shows up as a non-canonical value.
#include <cuda_runtime.h>

#include <cstdint>
#include <cstring>
#include <vector>

#include "ctx.hpp"
#include "marlin/poly.hpp"
#include "marlin/rng.hpp"
#include "marlin_ops.hpp"
#include "polyops.hpp"

using swb::Fr;

namespace {

swb_ctx* g_ctx = nullptr;

// device buffer freed at scope exit
struct DevBuf {
    void* p = nullptr;
    ~DevBuf() { if (p) cudaFree(p); }
};

int upload(DevBuf& d, const void* host, size_t bytes) {
    if (cudaMalloc(&d.p, bytes ? bytes : 32) != cudaSuccess) return -1;
    if (host && bytes && cudaMemcpyAsync(d.p, host, bytes, cudaMemcpyHostToDevice, g_ctx->stream) != cudaSuccess) return -1;
    return 0;
}
int alloc_poisoned(DevBuf& d, size_t bytes) {
    if (cudaMalloc(&d.p, bytes ? bytes : 32) != cudaSuccess) return -1;
    return cudaMemsetAsync(d.p, 0xFF, bytes ? bytes : 32, g_ctx->stream) == cudaSuccess ? 0 : -1;
}
int download(void* host, const DevBuf& d, size_t bytes) {
    if (bytes && cudaMemcpyAsync(host, d.p, bytes, cudaMemcpyDeviceToHost, g_ctx->stream) != cudaSuccess) return -1;
    return cudaStreamSynchronize(g_ctx->stream) == cudaSuccess ? 0 : -1;
}
Fr ld(const uint64_t* limbs) {
    Fr r;
    memcpy(r.l, limbs, sizeof(Fr));
    return r;
}
void st(uint64_t* limbs, const Fr& v) { memcpy(limbs, v.l, sizeof(Fr)); }

}  // namespace

#define EO_TRY(x)                  \
    do {                           \
        int rc__ = (x);            \
        if (rc__ != 0) return rc__; \
    } while (0)

extern "C" {

int eo_init(int device) {
    if (g_ctx) return 0;
    return swb_init(device, &g_ctx);
}
void eo_destroy() {
    if (g_ctx) swb_destroy(g_ctx);
    g_ctx = nullptr;
}
const char* eo_last_error() { return swb_last_error(g_ctx); }
int eo_sm_count() { return g_ctx ? g_ctx->sm_count : 0; }

// op: 0 a*=b, 1 a+=b, 2 a-=b, 3 a+=c0*b, 4 a*=c0, 5 a=c0+c1*a  (a is overwritten with the result)
int eo_poly_ew(int op, uint64_t* a, const uint64_t* b, size_t n, const uint64_t* c0, const uint64_t* c1) {
    DevBuf da, db;
    EO_TRY(upload(da, a, n * sizeof(Fr)));
    if (op <= 3) EO_TRY(upload(db, b, n * sizeof(Fr)));
    Fr* pa = (Fr*)da.p;
    const Fr* pb = (const Fr*)db.p;
    int rc;
    switch (op) {
        case 0: rc = swb::poly_mul_ew(g_ctx, pa, pb, n); break;
        case 1: rc = swb::poly_add_ew(g_ctx, pa, pb, n); break;
        case 2: rc = swb::poly_sub_ew(g_ctx, pa, pb, n); break;
        case 3: rc = swb::poly_add_scaled_ew(g_ctx, pa, ld(c0), pb, n); break;
        case 4: rc = swb::poly_scale_ew(g_ctx, pa, ld(c0), n); break;
        case 5: rc = swb::poly_lin_ew(g_ctx, pa, ld(c0), ld(c1), n); break;
        default: return SWB_EARG;
    }
    EO_TRY(rc);
    return download(a, da, n * sizeof(Fr));
}

int eo_poly_eval(const uint64_t* p, size_t n, const uint64_t* x, uint64_t* out) {
    DevBuf dp;
    EO_TRY(upload(dp, p, n * sizeof(Fr)));
    Fr r;
    EO_TRY(swb::poly_eval_dev(g_ctx, (const Fr*)dp.p, n, ld(x), &r));
    st(out, r);
    return 0;
}

// q: max(len - n, 0) elements, r: n elements
int eo_poly_div_vanishing(uint64_t* q, uint64_t* r, const uint64_t* p, size_t len, size_t n) {
    const size_t qlen = len > n ? len - n : 0;
    DevBuf dp, dq, dr;
    EO_TRY(upload(dp, p, len * sizeof(Fr)));
    EO_TRY(alloc_poisoned(dq, qlen * sizeof(Fr)));
    EO_TRY(alloc_poisoned(dr, n * sizeof(Fr)));
    EO_TRY(swb::poly_div_vanishing_dev(g_ctx, (Fr*)dq.p, (Fr*)dr.p, (const Fr*)dp.p, len, n));
    EO_TRY(download(q, dq, qlen * sizeof(Fr)));
    return download(r, dr, n * sizeof(Fr));
}

// q: n - 1 elements (n >= 2)
int eo_poly_div_linear(uint64_t* q, const uint64_t* p, size_t n, const uint64_t* z) {
    const size_t qlen = n > 1 ? n - 1 : 0;
    DevBuf dp, dq;
    EO_TRY(upload(dp, p, n * sizeof(Fr)));
    EO_TRY(alloc_poisoned(dq, qlen * sizeof(Fr)));
    EO_TRY(swb::poly_div_linear_dev(g_ctx, (Fr*)dq.p, (const Fr*)dp.p, n, ld(z)));
    return download(q, dq, qlen * sizeof(Fr));
}

int eo_poly_len(const uint64_t* p, size_t n, size_t* len) {
    DevBuf dp;
    EO_TRY(upload(dp, p, n * sizeof(Fr)));
    return swb::poly_len_dev(g_ctx, (const Fr*)dp.p, n, len);
}

int eo_poly_powers(uint64_t* out, size_t n, const uint64_t* g) {
    DevBuf d;
    EO_TRY(alloc_poisoned(d, n * sizeof(Fr)));
    EO_TRY(swb::poly_powers_dev(g_ctx, (Fr*)d.p, n, ld(g)));
    return download(out, d, n * sizeof(Fr));
}

int eo_rand_fr(uint64_t* out, size_t n, const uint32_t key[8], int rounds, uint64_t pos, uint64_t* words_used) {
    DevBuf d;
    EO_TRY(alloc_poisoned(d, n * sizeof(Fr)));
    EO_TRY(swb::rand_fr_dev(g_ctx, (Fr*)d.p, n, key, rounds, pos, words_used));
    return download(out, d, n * sizeof(Fr));
}

// start: nrows + 1 offsets; col / coef / tag: start[nrows] entries; tag and weights may be NULL
int eo_csr_spmv(uint64_t* out, size_t nout, size_t nrows, const uint32_t* start, const uint32_t* col, const uint64_t* coef,
                const uint8_t* tag, const uint64_t* x, size_t xlen, const uint64_t* weights) {
    const size_t nnz = start[nrows];
    DevBuf dout, dstart, dcol, dcoef, dtag, dx;
    EO_TRY(alloc_poisoned(dout, nout * sizeof(Fr)));
    EO_TRY(upload(dstart, start, (nrows + 1) * sizeof(uint32_t)));
    EO_TRY(upload(dcol, col, nnz * sizeof(uint32_t)));
    EO_TRY(upload(dcoef, coef, nnz * sizeof(Fr)));
    if (tag) EO_TRY(upload(dtag, tag, nnz));
    EO_TRY(upload(dx, x, xlen * sizeof(Fr)));
    Fr w[3];
    if (weights)
        for (int i = 0; i < 3; i++) w[i] = ld(weights + 4 * i);
    EO_TRY(swb::csr_spmv_dev(g_ctx, (Fr*)dout.p, nout, nrows, (const uint32_t*)dstart.p, (const uint32_t*)dcol.p, (const Fr*)dcoef.p,
                             tag ? (const uint8_t*)dtag.p : nullptr, (const Fr*)dx.p, weights ? w : nullptr));
    return download(out, dout, nout * sizeof(Fr));
}

// z: nvars elements, xh: nh elements
int eo_witness_evals(uint64_t* out, size_t nh, size_t ratio, const uint64_t* z, size_t ninst, size_t nvars, const uint64_t* xh) {
    DevBuf dout, dz, dxh;
    EO_TRY(alloc_poisoned(dout, nh * sizeof(Fr)));
    EO_TRY(upload(dz, z, nvars * sizeof(Fr)));
    EO_TRY(upload(dxh, xh, nh * sizeof(Fr)));
    EO_TRY(swb::witness_evals_dev(g_ctx, (Fr*)dout.p, nh, ratio, (const Fr*)dz.p, ninst, nvars, (const Fr*)dxh.p));
    return download(out, dout, nh * sizeof(Fr));
}

// ---- the host engine's versions (the CPU arm's arithmetic), references past python-integer sizes ----
void eo_host_poly_eval(const uint64_t* p, size_t n, const uint64_t* x, uint64_t* out) {
    swb::marlin::Poly v((const Fr*)p, (const Fr*)p + n);
    st(out, swb::marlin::poly_eval(v, ld(x)));
}

void eo_host_poly_div_vanishing(uint64_t* q, uint64_t* r, const uint64_t* p, size_t len, size_t n) {
    swb::marlin::Poly v((const Fr*)p, (const Fr*)p + len), qq, rr;
    swb::marlin::poly_divide_by_vanishing(v, n, &qq, &rr);
    memcpy(q, qq.data(), qq.size() * sizeof(Fr));
    memcpy(r, rr.data(), rr.size() * sizeof(Fr));
}

void eo_host_poly_div_linear(uint64_t* q, const uint64_t* p, size_t n, const uint64_t* z) {
    swb::marlin::Poly v((const Fr*)p, (const Fr*)p + n);
    swb::marlin::Poly qq = swb::marlin::poly_divide_by_linear(v, ld(z));
    memcpy(q, qq.data(), qq.size() * sizeof(Fr));
}

void eo_host_rand_fr(uint64_t* out, size_t n, const uint32_t key[8], int rounds, uint64_t pos, uint64_t* words_used) {
    uint8_t seed[32];
    for (int i = 0; i < 8; i++)
        for (int b = 0; b < 4; b++) seed[4 * i + b] = (uint8_t)(key[i] >> (8 * b));
    swb::marlin::ChaChaRng rng(seed, rounds);
    rng.seek(pos);
    swb::marlin::rand_fr_bulk(rng, (Fr*)out, n);
    *words_used = rng.position() - pos;
}

}  // extern "C"
