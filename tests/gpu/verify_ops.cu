// Test-only shim: the batch verifier's point decoder (verify_ops.hpp: g1_decode_dev, the kernel k_g1_decode) and the
// host parser's decoder (marlin/curve_host.hpp: get_g1_compressed) behind plain extern "C" functions, so that
// tests/test_gpu_verify_batch.py can compare them encoding by encoding through ctypes.
#include <cuda_runtime.h>

#include <cstdint>
#include <cstring>

#include "ctx.hpp"
#include "marlin/curve_host.hpp"
#include "verify_ops.hpp"

namespace {
swb_ctx* g_ctx = nullptr;
struct DevBuf {
    void* p = nullptr;
    ~DevBuf() { if (p) cudaFree(p); }
};
}  // namespace

extern "C" {

int vo_init(int device) { return swb_init(device, &g_ctx); }
void vo_destroy(void) {
    swb_destroy(g_ctx);
    g_ctx = nullptr;
}
const char* vo_last_error(void) { return swb_last_error(g_ctx); }

// n encodings of 48 bytes -> xy (n x 96 bytes: Montgomery x | y, (0, 0) for the identity and for refused encodings) and
// status (g1_decode's G1DecodeStatus) from the kernel.  The outputs are filled with 0xFF bytes before the launch.
int vo_decode_dev(const uint8_t* enc, size_t n, uint8_t* xy, uint8_t* status) {
    DevBuf e, o, s;
    if (cudaMalloc(&e.p, n * 48 + 64) != cudaSuccess || cudaMalloc(&o.p, n * 96 + 64) != cudaSuccess ||
        cudaMalloc(&s.p, n + 64) != cudaSuccess)
        return SWB_ENOMEM;
    cudaStream_t st = g_ctx->stream;
    if (cudaMemcpyAsync(e.p, enc, n * 48, cudaMemcpyHostToDevice, st) != cudaSuccess ||
        cudaMemsetAsync(o.p, 0xFF, n * 96, st) != cudaSuccess || cudaMemsetAsync(s.p, 0xFF, n, st) != cudaSuccess)
        return SWB_ECUDA;
    int rc = swb::g1_decode_dev(g_ctx, static_cast<const uint32_t*>(e.p), n, swb::marlin::g1_decode_consts(), static_cast<swb::Fq*>(o.p),
                                static_cast<uint8_t*>(s.p));
    if (rc != SWB_OK) return rc;
    if (cudaMemcpyAsync(xy, o.p, n * 96, cudaMemcpyDeviceToHost, st) != cudaSuccess ||
        cudaMemcpyAsync(status, s.p, n, cudaMemcpyDeviceToHost, st) != cudaSuccess || cudaStreamSynchronize(st) != cudaSuccess)
        return SWB_ECUDA;
    return SWB_OK;
}

// the same encodings through the host parser: ok[i] = get_g1_compressed's verdict, xy as above (zeros when refused)
void vo_decode_host(const uint8_t* enc, size_t n, uint8_t* xy, uint8_t* ok) {
#pragma omp parallel for schedule(dynamic, 64)
    for (long i = 0; i < (long)n; i++) {
        const uint8_t* p = enc + 48 * i;
        swb::marlin::G1Point pt;
        ok[i] = swb::marlin::get_g1_compressed(p, enc + 48 * (i + 1), &pt) ? 1 : 0;
        const swb::Fq zero = swb::Fq::zero();
        memcpy(xy + 96 * i, (ok[i] && !pt.infinity ? pt.x : zero).l, 48);
        memcpy(xy + 96 * i + 48, (ok[i] && !pt.infinity ? pt.y : zero).l, 48);
    }
}

}  // extern "C"
