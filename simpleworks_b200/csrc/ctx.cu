// Context, error reporting, device buffers.
#include <algorithm>
#include <cstdarg>
#include <cstdlib>
#include <cstring>
#include <mutex>

#include "ctx.hpp"

namespace {
std::mutex g_init_mu;
std::string g_init_err;
}  // namespace

namespace swb {

int set_err(swb_ctx* c, int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (c) c->err = buf;
    else {
        std::lock_guard<std::mutex> g(g_init_mu);
        g_init_err = buf;
    }
    return code;
}

int cuda_fail(swb_ctx* c, cudaError_t e, const char* what) {
    return set_err(c, SWB_ECUDA, "CUDA error %d (%s) at %s", (int)e, cudaGetErrorString(e), what);
}

void sync_all_streams(swb_ctx* c) {
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    for (auto& sl : c->msm_slot) {
        if (sl.work) cudaStreamSynchronize(sl.work);
        if (sl.tail) cudaStreamSynchronize(sl.tail);
    }
}

void* vec_alloc(swb_ctx* c, size_t bytes, size_t* granted) {
    const size_t unit = (size_t)2 << 20;
    const size_t want = bytes ? (bytes + unit - 1) / unit * unit : unit;
    auto it = c->vec_cache.lower_bound(want);
    if (it != c->vec_cache.end() && it->first <= want + want / 4) {      // close fit: do not burn a big block on a small vector
        void* p = it->second;
        *granted = it->first;
        c->vec_cache_bytes -= it->first;
        c->vec_cache.erase(it);
        return p;
    }
    void* p = nullptr;
    cudaError_t e = cudaMalloc(&p, want);
    if (e != cudaSuccess) {
        // out of memory: give the cache back and retry once
        cudaGetLastError();
        cudaStreamSynchronize(c->stream);
        for (auto& kv : c->vec_cache) cudaFree(kv.second);
        c->vec_cache.clear();
        c->vec_cache_bytes = 0;
        e = cudaMalloc(&p, want);
        if (e != cudaSuccess) {
            cudaGetLastError();
            set_err(c, SWB_ENOMEM, "vec_alloc: cudaMalloc(%zu) failed: %s", want, cudaGetErrorString(e));
            return nullptr;
        }
    }
    *granted = want;
    return p;
}
void vec_free(swb_ctx* c, void* p, size_t granted) {
    if (!p) return;
    c->vec_cache.emplace(granted, p);
    c->vec_cache_bytes += granted;
    // a prover that keeps changing sizes must not hoard the device: past a third of its memory the cache
    // is handed back (after the stream has drained, since cached blocks may still be in use on it)
    if (c->total_mem && c->vec_cache_bytes > c->total_mem / 3) {
        cudaSetDevice(c->device);
        cudaStreamSynchronize(c->stream);
        for (auto& kv : c->vec_cache) cudaFree(kv.second);
        c->vec_cache.clear();
        c->vec_cache_bytes = 0;
    }
}

void* get_scratch(swb_ctx* c, const char* tag, size_t bytes) {
    auto& s = c->scratch_slot ? c->scratch[std::string(tag) + "#" + std::to_string(c->scratch_slot)] : c->scratch[tag];
    if (s.bytes >= bytes && s.p) return s.p;
    if (s.p) {
        cudaStreamSynchronize(c->stream);
        cudaFree(s.p);
        s.p = nullptr;
        s.bytes = 0;
    }
    size_t want = bytes + bytes / 8 + 256;
    cudaError_t e = cudaMalloc(&s.p, want);
    if (e != cudaSuccess) {
        s.p = nullptr;
        set_err(c, SWB_ENOMEM, "cudaMalloc(%zu) for scratch '%s' failed: %s", want, tag, cudaGetErrorString(e));
        return nullptr;
    }
    s.bytes = want;
    return s.p;
}

void* get_pinned(swb_ctx* c, size_t bytes) {
    if (c->pinned_bytes >= bytes && c->pinned) return c->pinned;
    if (c->pinned) cudaFreeHost(c->pinned);
    c->pinned = nullptr;
    c->pinned_bytes = 0;
    if (cudaMallocHost(&c->pinned, bytes) != cudaSuccess) {
        c->pinned = nullptr;
        set_err(c, SWB_ENOMEM, "cudaMallocHost(%zu) failed", bytes);
        return nullptr;
    }
    c->pinned_bytes = bytes;
    return c->pinned;
}

}  // namespace swb

extern "C" {

int swb_init(int device, swb_ctx** out) {
    if (!out) return swb::set_err(nullptr, SWB_EARG, "swb_init: out is NULL");
    *out = nullptr;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return swb::set_err(nullptr, SWB_ECUDA,
                            "swb_init: no CUDA device (%s); libswb200 has no CPU fallback",
                            e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
    if (device < 0 || device >= ndev) return swb::set_err(nullptr, SWB_EARG, "swb_init: device %d out of range [0,%d)", device, ndev);
    e = cudaSetDevice(device);
    if (e != cudaSuccess) return swb::cuda_fail(nullptr, e, "cudaSetDevice");
    cudaDeviceProp prop;
    e = cudaGetDeviceProperties(&prop, device);
    if (e != cudaSuccess) return swb::cuda_fail(nullptr, e, "cudaGetDeviceProperties");
    if (prop.major != 10)
        return swb::set_err(nullptr, SWB_ECUDA, "swb_init: device %d is sm_%d%d; this library is built for sm_100a only", device,
                            prop.major, prop.minor);
    swb_ctx* c = new swb_ctx();
    c->device = device;
    c->sm_count = prop.multiProcessorCount;
    c->cc_major = prop.major;
    c->cc_minor = prop.minor;
    c->total_mem = prop.totalGlobalMem;
    e = cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) {
        delete c;
        return swb::cuda_fail(nullptr, e, "cudaStreamCreate");
    }
    c->stream = c->own_stream;
    const char* tr = getenv("SWB_TRACE");
    c->trace = tr ? atoi(tr) : 0;
    int rc = swb::ntt_build_tables(c);
    if (rc != SWB_OK) {
        swb::set_err(nullptr, rc, "%s", c->err.c_str());
        swb_destroy(c);
        return rc;
    }
    *out = c;
    return SWB_OK;
}

void swb_destroy(swb_ctx* c) {
    if (!c) return;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    swb_comm_destroy(c);
    // unlink from the peer relation on both sides, whichever context goes first
    for (swb_ctx* p : c->msm_peers) p->msm_primaries.erase(std::find(p->msm_primaries.begin(), p->msm_primaries.end(), c));
    for (swb_ctx* q : c->msm_primaries) q->msm_peers.erase(std::find(q->msm_peers.begin(), q->msm_peers.end(), c));
    if (c->peer_ev) cudaEventDestroy(c->peer_ev);
    for (auto& kv : c->vec_cache) cudaFree(kv.second);
    for (auto& sl : c->msm_slot) {
        if (sl.work) { cudaStreamSynchronize(sl.work); cudaStreamDestroy(sl.work); }
        if (sl.tail) { cudaStreamSynchronize(sl.tail); cudaStreamDestroy(sl.tail); }
        if (sl.ev) cudaEventDestroy(sl.ev);
        if (sl.host_wins) cudaFreeHost(sl.host_wins);
    }
    for (auto& kv : c->scratch)
        if (kv.second.p) cudaFree(kv.second.p);
    if (c->pinned) cudaFreeHost(c->pinned);
    if (c->pair_count_host) cudaFreeHost(c->pair_count_host);
    if (c->tw_root) cudaFree(c->tw_root);
    if (c->tw_gen) cudaFree(c->tw_gen);
    if (c->tw_geninv) cudaFree(c->tw_geninv);
    if (c->tw_full) cudaFree(c->tw_full);
    if (c->own_stream) cudaStreamDestroy(c->own_stream);
    delete c;
}

int swb_trim(swb_ctx* c) {
    if (!c) return SWB_EARG;
    for (auto& sl : c->msm_slot)
        if (sl.active) return swb::set_err(c, SWB_EARG, "trim: an MSM is still in flight");
    cudaSetDevice(c->device);
    swb::sync_all_streams(c);
    for (auto& kv : c->scratch)
        if (kv.second.p) cudaFree(kv.second.p);
    c->scratch.clear();
    for (auto& kv : c->vec_cache) cudaFree(kv.second);
    c->vec_cache.clear();
    c->vec_cache_bytes = 0;
    if (c->tw_full) cudaFree(c->tw_full);
    c->tw_full = nullptr;
    c->tw_full_log = 0;
    c->tw_full_failed = false;
    return SWB_OK;
}

const char* swb_last_error(const swb_ctx* c) {
    if (c) return c->err.c_str();
    std::lock_guard<std::mutex> g(g_init_mu);
    static thread_local std::string copy;
    copy = g_init_err;
    return copy.c_str();
}

int swb_set_stream(swb_ctx* c, void* s) {
    if (!c) return SWB_EARG;
    // scratch and cached blocks are reused in stream order: drain the old stream before work moves
    if (c->stream != (cudaStream_t)s) {
        cudaSetDevice(c->device);
        cudaStreamSynchronize(c->stream);
    }
    c->stream = (cudaStream_t)s;
    return SWB_OK;
}

int swb_reset_stream(swb_ctx* c) {
    if (!c) return SWB_EARG;
    c->stream = c->own_stream;
    return SWB_OK;
}

int swb_sync(swb_ctx* c) {
    if (!c) return SWB_EARG;
    SWB_CUDA(c, cudaStreamSynchronize(c->stream));
    return SWB_OK;
}

int swb_device_info(swb_ctx* c, int* sm_count, int* cc_major, int* cc_minor, size_t* total_mem) {
    if (!c) return SWB_EARG;
    if (sm_count) *sm_count = c->sm_count;
    if (cc_major) *cc_major = c->cc_major;
    if (cc_minor) *cc_minor = c->cc_minor;
    if (total_mem) *total_mem = c->total_mem;
    return SWB_OK;
}

uint64_t swb_launch_count(const swb_ctx* c) { return c ? c->launches : 0; }

int swb_profile_enable(swb_ctx* c, int enable) {
    if (!c) return SWB_EARG;
    c->profile = enable ? 1 : 0;
    return SWB_OK;
}

int swb_profile_last(swb_ctx* c, const char** names, double* ms, int cap, int* count) {
    if (!c || !count) return SWB_EARG;
    int k = 0;
    for (auto& st : c->last_stages) {
        if (k >= cap) break;
        if (names) names[k] = st.first;
        if (ms) ms[k] = st.second;
        k++;
    }
    *count = k;
    return SWB_OK;
}

int swb_dev_alloc(swb_ctx* c, size_t bytes, void** out) {
    if (!c || !out) return SWB_EARG;
    SWB_CUDA(c, cudaSetDevice(c->device));
    cudaError_t e = cudaMalloc(out, bytes ? bytes : 1);
    if (e != cudaSuccess) return swb::set_err(c, SWB_ENOMEM, "cudaMalloc(%zu): %s", bytes, cudaGetErrorString(e));
    return SWB_OK;
}
int swb_dev_free(swb_ctx* c, void* p) {
    if (!c) return SWB_EARG;
    SWB_CUDA(c, cudaStreamSynchronize(c->stream));
    SWB_CUDA(c, cudaFree(p));
    return SWB_OK;
}
int swb_h2d(swb_ctx* c, void* dst, const void* src, size_t bytes) {
    if (!c) return SWB_EARG;
    SWB_CUDA(c, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, c->stream));
    SWB_CUDA(c, cudaStreamSynchronize(c->stream));
    return SWB_OK;
}
int swb_d2h(swb_ctx* c, void* dst, const void* src, size_t bytes) {
    if (!c) return SWB_EARG;
    SWB_CUDA(c, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, c->stream));
    SWB_CUDA(c, cudaStreamSynchronize(c->stream));
    return SWB_OK;
}

}  // extern "C"
