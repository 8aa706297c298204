// Test-only shim: the Marlin engine of marlin_abi.cu (included whole, so that its internal GpuEngine is reachable) on a
// context of the shim's own with peer contexts on the same device.  It makes a call fail while the peers hold shares
// -- requests noted or running on their slots, scalar copies in their vector caches -- and checks what msm_abandon
// leaves behind (tests/test_gpu_msm_peers_abandon.py).
#include "marlin_abi.cu"

namespace {
swb_ctx* g_ctx = nullptr;
std::vector<swb_ctx*> g_peers;
}  // namespace

extern "C" {

int pa_init(int n_peers) {
    int rc = swb_init(0, &g_ctx);
    for (int i = 0; i < n_peers && rc == SWB_OK; i++) {
        swb_ctx* p = nullptr;
        rc = swb_init(0, &p);
        if (rc == SWB_OK) g_peers.push_back(p);
    }
    return rc == SWB_OK ? swb_set_msm_peers(g_ctx, g_peers.data(), (int)g_peers.size()) : rc;
}
void pa_destroy(void) {
    swb_destroy(g_ctx);
    for (swb_ctx* p : g_peers) swb_destroy(p);
    g_ctx = nullptr;
    g_peers.clear();
}

// Submits four sharded MSMs of about n scalars over beta^i * g (window tables of `window_bits` when > 0), launches the
// peers' queues as combine_pending would, then abandons.  Afterwards every peer must hold no request and no busy slot,
// its scalar copies must be back in its vector cache, every context must trim, and the engine's next MSM must equal
// the unsharded one (swb_msm_g1_fr on the context, which swb_set_msm_peers does not share).  Returns 0, or the number of
// the check that failed (message in msg).
int pa_abandon_check(const swb_g1_jacobian* g, const swb_fr* beta, size_t n, int window_bits, const swb_fr* scalars, char* msg,
                     size_t cap) {
    swb_bases* b = nullptr;
    if (swb_bases_from_powers(g_ctx, g, beta, n, &b) != SWB_OK) return 1;
    if (window_bits > 0 && swb_bases_precompute(g_ctx, b, window_bits) != SWB_OK) return 2;
    int step = 3;
    GpuEngine eng(g_ctx);
    try {
        std::vector<Fr> h(n);
        memcpy(h.data(), scalars, n * sizeof(Fr));
        GpuEngine::Vec v = eng.vfrom(h);
        for (int k = 0; k < 4; k++) eng.msm_submit(b, 0, v, n - 97 * k);
        step = 4;
        size_t noted = 0;
        for (swb_ctx* p : g_peers) {
            bool launched = false;
            if (msm_queue_launch(p, &launched) != SWB_OK) throw MarlinError(swb_last_error(p));
            noted += p->msm_queue.size();
        }
        if (noted == 0) { snprintf(msg, cap, "the peers hold no shares"); return step; }
        eng.msm_abandon();
        step = 5;
        for (swb_ctx* p : g_peers) {
            bool busy = !p->msm_queue.empty();
            for (auto& sl : p->msm_slot) busy |= sl.active;
            if (busy) { snprintf(msg, cap, "a peer still holds a request or a busy slot"); return step; }
            if (p->vec_cache_bytes == 0) { snprintf(msg, cap, "a peer's scalar copy was not returned to its cache"); return step; }
        }
        step = 6;
        if (swb_trim(g_ctx) != SWB_OK) { snprintf(msg, cap, "trim: %s", swb_last_error(g_ctx)); return step; }
        for (swb_ctx* p : g_peers)
            if (swb_trim(p) != SWB_OK) { snprintf(msg, cap, "trim (peer): %s", swb_last_error(p)); return step; }
        step = 7;
        const G1Point got = eng.msm_result(eng.msm_submit(b, 0, v, n));
        swb_g1_jacobian want;
        if (swb_msm_g1_fr(g_ctx, b, 0, scalars, n, &want) != SWB_OK) throw MarlinError(swb_last_error(g_ctx));
        step = 8;
        if (got.infinity || memcmp(got.x.l, want.x.l, 48) != 0 || memcmp(got.y.l, want.y.l, 48) != 0) {
            snprintf(msg, cap, "the MSM after the abandon differs from the unsharded one");
            return step;
        }
        v.release();
        eng.free_bases(b);
        return 0;
    } catch (const std::exception& e) {
        snprintf(msg, cap, "%s", e.what());
        return 100 + step;
    }
}

}  // extern "C"
