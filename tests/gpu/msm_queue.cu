// Test-only shim: the context's MSM queue (ctx.hpp: msm_queue_*) behind plain extern "C" functions on a context of the
// shim's own, with the few ABI calls tests/test_gpu_msm_queue.py needs around it (bases, single MSMs, trim).
#include <cuda_runtime.h>

#include <cstdint>

#include "ctx.hpp"

namespace {
swb_ctx* g_ctx = nullptr;
}  // namespace

extern "C" {

int mq_init(int device) {
    int rc = swb_init(device, &g_ctx);
    // tables whenever the bases have them, so that small requests batch
    return rc == SWB_OK ? swb_msm_set_table_policy(g_ctx, 1) : rc;
}
void mq_destroy(void) {
    swb_destroy(g_ctx);
    g_ctx = nullptr;
}
const char* mq_last_error(void) { return swb_last_error(g_ctx); }
uint64_t mq_launch_count(void) { return swb_launch_count(g_ctx); }
int mq_trim(void) { return swb_trim(g_ctx); }

// bases beta^i * g, i < n, with window tables of `window_bits` when it is > 0
swb_bases* mq_bases(const swb_g1_jacobian* g, const swb_fr* beta, size_t n, int window_bits) {
    swb_bases* b = nullptr;
    if (swb_bases_from_powers(g_ctx, g, beta, n, &b) != SWB_OK) return nullptr;
    if (window_bits > 0 && swb_bases_precompute(g_ctx, b, window_bits) != SWB_OK) {
        swb_bases_free(b);
        return nullptr;
    }
    return b;
}
void mq_bases_free(swb_bases* b) { swb_bases_free(b); }

void* mq_upload(const void* host, size_t bytes) {
    void* d = nullptr;
    if (cudaMalloc(&d, bytes ? bytes : 32) != cudaSuccess) return nullptr;
    if (bytes && cudaMemcpy(d, host, bytes, cudaMemcpyHostToDevice) != cudaSuccess) {
        cudaFree(d);
        return nullptr;
    }
    return d;
}
void mq_free(void* d) { cudaFree(d); }

// the single call (swb_msm_g1_dev / swb_msm_g1_fr_dev) under bucket shard (rank, world)
int mq_single(const swb_bases* b, size_t offset, const void* scalars_dev, size_t n, int montgomery, int rank, int world,
              swb_g1_jacobian* out) {
    int rc = swb_msm_set_bucket_shard(g_ctx, rank, world);
    if (rc != SWB_OK) return rc;
    rc = montgomery ? swb_msm_g1_fr_dev(g_ctx, b, offset, static_cast<const swb_fr*>(scalars_dev), n, out)
                    : swb_msm_g1_dev(g_ctx, b, offset, static_cast<const swb_bigint256*>(scalars_dev), n, out);
    swb_msm_set_bucket_shard(g_ctx, 0, 1);
    return rc;
}

int mq_submit(const swb_bases* b, size_t offset, const void* scalars_dev, size_t n, int montgomery, int rank, int world, size_t* id) {
    return swb::msm_queue_submit(g_ctx, b, offset, scalars_dev, n, montgomery, swb::BucketShard{rank, world}, id);
}
int mq_flush(void) { return swb::msm_queue_flush(g_ctx); }
int mq_result(size_t id, swb_g1_jacobian* out) { return swb::msm_queue_result(g_ctx, id, out); }
void mq_abandon(void) { swb::msm_queue_abandon(g_ctx); }
// MSM slots that hold a launched MSM
int mq_active_slots(void) {
    int k = 0;
    for (auto& sl : g_ctx->msm_slot) k += sl.active ? 1 : 0;
    return k;
}

}  // extern "C"
