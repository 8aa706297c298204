// Internal context shared by the translation units of libswb200.
#pragma once
#include <cuda_runtime.h>

#include <cstdint>
#include <cstdio>
#include <map>
#include <string>
#include <vector>

#include "../../include/swb200.h"
#include "fp.cuh"

namespace swb {
// A bucket shard: the MSM fills only the buckets b with b mod world == rank of every bucket set and returns that share of
// the result (world a power of two; world = 1: all buckets)
struct BucketShard { int rank, world; };
}  // namespace swb

struct swb_ctx {
    int device = 0;
    int sm_count = 0;
    int cc_major = 0, cc_minor = 0;
    size_t total_mem = 0;
    cudaStream_t own_stream = nullptr;
    cudaStream_t stream = nullptr;
    std::string err;
    uint64_t launches = 0;
    int msm_window_override = 0;
    int msm_pair_policy = 1;   // swb_msm_set_pair_sums: batch-affine pair sums before the accumulation (0 never, 1 automatic, 2 always)
    int msm_table_policy = 0;  // swb_msm_set_table_policy: -1 never, 0 automatic, 1 whenever the bases have tables
    int trace = 0;            // SWB_TRACE=1: per-stage CUDA-event timings on stderr
    int profile = 0;          // swb_profile_enable: keep the last call's stage timings
    std::vector<std::pair<const char*, double>> last_stages;

    // NTT tables (device): three levels of 1024 powers of the 2^30-th root of unity, and of the
    // coset generator 22 and its inverse.  Built by one kernel at swb_init.
    swb::Fr* tw_root = nullptr;   // [3][1024]
    swb::Fr* tw_gen = nullptr;    // [3][1024]
    swb::Fr* tw_geninv = nullptr; // [3][1024]
    swb::Fr* tw_full = nullptr;   // [2^tw_full_log] powers of the 2^tw_full_log-th root of unity (inter-digit twiddles by direct lookup)
    uint32_t tw_full_log = 0;
    bool tw_full_failed = false;  // allocation refused once: stay on running products

    // grow-only scratch arena so repeated calls do not cudaMalloc in the timed path
    struct Scratch { void* p = nullptr; size_t bytes = 0; };
    std::map<std::string, Scratch> scratch;
    void* pinned = nullptr;
    size_t pinned_bytes = 0;
    uint32_t* pair_count_host = nullptr;   // pinned word: summed slots of the last pair-sum pass (profiling)

    // MSM slots: slot 0 runs on `stream` (the swb_msm_* single calls and the queue's batches); slots 1..MSM_SLOTS-1
    // have streams of their own (a normal one for sort + accumulation, a high-priority one for the latency-bound
    // bucket tail) and their own scratch, so that the queue's independent MSMs overlap.  Only msm.cu starts and
    // finishes MSMs on them.
    static constexpr int MSM_SLOTS = 3;
    struct MsmSlot {
        cudaStream_t work = nullptr, tail = nullptr;
        cudaEvent_t ev = nullptr;
        void* host_wins = nullptr;     // pinned, MSM_MAX_WINDOWS XYZZ points
        int nwin = 0, cb = 0;
        int nres = 1;                  // results the slot will deliver (vectors of a batch)
        bool batched = false;          // one bucket set per vector, no Horner fold
        int shard_rank = 0, shard_world = 1;   // bucket shard this MSM was planned for (swb_msm_set_bucket_shard)
        bool active = false, empty = false;
    } msm_slot[MSM_SLOTS];
    int scratch_slot = 0;              // suffix of scratch tags while a slot > 0 is being launched
    // the MSM queue (msm_queue_* below): requests by id, from submission until their result is taken
    struct MsmRequest {
        const swb_bases* bases; size_t offset, n; const void* scalars; int montgomery; swb::BucketShard shard;
        int slot = -1;                 // -1: noted; else the slot it was launched on
        bool single = false;           // noted, and its run could not go out as one batch: launched on its own
        bool done = false;             // finished: the result is in `out`
        swb_g1_jacobian out;
    };
    std::map<size_t, MsmRequest> msm_queue;
    size_t msm_queue_next = 0;         // id of the next request
    int msm_next_slot = 1;             // slot of the next single MSM (1 and 2 alternately)
    // bucket sharding of the swb_msm_* entry points (swb_msm_set_bucket_shard, swb::BucketShard)
    int bucket_rank = 0, bucket_world = 1;
    // multi-GPU proving (swb_set_msm_shard): this rank's share of every prover MSM, and who adds them up
    int shard_rank = 0, shard_world = 1;
    int (*shard_combine)(void*, const swb_g1_jacobian*, swb_g1_jacobian*) = nullptr;
    void* shard_user = nullptr;
    // swb_set_msm_peers: contexts of this process that take ranks 1..n of every prover MSM (this context is rank 0),
    // and the contexts that have this one as a peer (swb_destroy of either side unlinks it)
    std::vector<swb_ctx*> msm_peers;
    std::vector<swb_ctx*> msm_primaries;
    cudaEvent_t peer_ev = nullptr;     // orders a copy to a peer after the work queued on `stream`
    uint64_t peer_bytes = 0;           // bytes copied to the peers (swb_peer_copy_bytes)

    // swb_comm_*: NCCL communicator of this context (one process per GPU), staging buffers of the all-gather
    void* comm = nullptr;
    int comm_rank = 0, comm_world = 1;
    void *comm_dev = nullptr, *comm_host = nullptr;

    // cache of freed device blocks for the engine's vectors (vec_alloc / vec_free below), by size
    std::multimap<size_t, void*> vec_cache;
    size_t vec_cache_bytes = 0;
};

struct swb_bases {
    swb_ctx* ctx = nullptr;
    swb::Fq* xy = nullptr;   // n records of 96 bytes: x | y ; identity = (0,0)
    size_t n = 0;
    // window tables (swb_bases_precompute): xy then holds tab_w levels of n records,
    // level j = 2^(tab_c * j) * base
    int tab_c = 0, tab_w = 0;
};

namespace swb {

constexpr int MSM_MAX_BATCH = 16;   // MSMs that one batched call may hold (one bucket set each)

int set_err(swb_ctx* c, int code, const char* fmt, ...);
// wait for the context's stream and for the MSM slots' own streams (before device memory they may be
// reading is released)
void sync_all_streams(swb_ctx* c);
// The MSM queue: submission checks a request and only notes it (its scalars must stay alive until the result is taken
// or the queue abandoned).  A flush launches the noted requests: consecutive ones over the same bases, bucket shard and
// scalar form make runs of up to MSM_MAX_BATCH; a run of two or more over window tables goes out as ONE batched pipeline,
// every other request goes to slots 1 and 2 alternately, so that the bucket tail of one runs under the accumulation of
// the next.  A result is the affine value as a Z = 1 Jacobian (Z = 0, and n = 0: the identity).
int msm_queue_submit(swb_ctx* c, const swb_bases* bases, size_t offset, const void* scalars_dev, size_t n, int montgomery,
                     BucketShard shard, size_t* id);
int msm_queue_flush(swb_ctx* c);
// launches the next run of noted requests: a batch, or one request on the next slot of 1 and 2 once that slot's previous
// MSM has finished.  *launched = false when nothing is noted.  A flush launches until nothing is; a caller that drives
// several contexts launches a run on each in turn, so that their devices work at once.
int msm_queue_launch(swb_ctx* c, bool* launched);
// flushes when the request is still noted, waits for it and hands its result over (once)
int msm_queue_result(swb_ctx* c, size_t id, swb_g1_jacobian* out);
// launches and finishes every request, keeping the results (before the bases they read are replaced)
int msm_queue_drain(swb_ctx* c);
// waits for the launched requests, frees their slots and forgets every request (failure paths)
void msm_queue_abandon(swb_ctx* c);
// fixed_base.cu: the window-table width that suits MSMs of about n scalars (what swb_bases_precompute picks for
// window_bits = 0)
int tables_pick_window(size_t n);
// Device blocks for short-lived vectors (the prover allocates and frees hundreds per proof).  All work of
// a context is ordered on one stream, so a freed block can be handed to the next request at once;
// blocks are rounded to 2 MiB and kept until swb_destroy, which keeps cudaMalloc/cudaFree (and the
// driver's own pool maintenance) out of the steady state.  *granted is the block's real size, to be
// passed back to vec_free.  nullptr + error set on failure.
void* vec_alloc(swb_ctx* c, size_t bytes, size_t* granted);
void vec_free(swb_ctx* c, void* p, size_t granted);
int cuda_fail(swb_ctx* c, cudaError_t e, const char* what);
// comm.cu: out[k] = sum over the ranks of mine[k], k < count -- one all-gather on the context's stream
int comm_sum_g1(swb_ctx* c, const swb_g1_jacobian* mine, size_t count, swb_g1_jacobian* out);
// returns device scratch of at least `bytes`, tagged; nullptr + error set on failure
void* get_scratch(swb_ctx* c, const char* tag, size_t bytes);
void* get_pinned(swb_ctx* c, size_t bytes);

#define SWB_CUDA(ctx, call)                                                   \
    do {                                                                      \
        cudaError_t e__ = (call);                                             \
        if (e__ != cudaSuccess) return swb::cuda_fail((ctx), e__, #call);     \
    } while (0)

#define SWB_LAUNCH_CHECK(ctx, name)                                           \
    do {                                                                      \
        (ctx)->launches++;                                                    \
        cudaError_t e__ = cudaGetLastError();                                 \
        if (e__ != cudaSuccess) return swb::cuda_fail((ctx), e__, name);      \
    } while (0)

#define SWB_REQUIRE(ctx, cond, msg)                                           \
    do {                                                                      \
        if (!(cond)) return swb::set_err((ctx), SWB_EARG, "%s", msg);         \
    } while (0)

// per-stage CUDA-event timer, active only when ctx->trace is set
struct StageTimer {
    swb_ctx* c;
    const char* what;
    std::vector<std::pair<const char*, cudaEvent_t>> marks;
    // spans: kernels of one kind launched many times inside a stage (begin/end event pairs, summed per name)
    struct Span { const char* name; cudaEvent_t a, b; };
    std::vector<Span> spans;
    // counters: 32-bit values in pinned host memory that a copy queued on the stream fills; reported in millions
    std::vector<std::pair<const char*, const uint32_t*>> counters;
    void counter(const char* name, const uint32_t* host_value) { if (on()) counters.emplace_back(name, host_value); }
    StageTimer(swb_ctx* ctx, const char* w) : c(ctx), what(w) { mark("start"); }
    bool on() const { return c->trace || c->profile; }
    void span_begin(const char* name) {
        if (!on()) return;
        Span s{name, nullptr, nullptr};
        cudaEventCreate(&s.a);
        cudaEventCreate(&s.b);
        cudaEventRecord(s.a, c->stream);
        spans.push_back(s);
    }
    void span_end() {
        if (!on() || spans.empty()) return;
        cudaEventRecord(spans.back().b, c->stream);
    }
    void mark(const char* name) {
        if (!c->trace && !c->profile) return;
        cudaEvent_t e;
        cudaEventCreate(&e);
        cudaEventRecord(e, c->stream);
        marks.emplace_back(name, e);
    }
    ~StageTimer() {
        if ((!c->trace && !c->profile) || marks.empty()) return;
        cudaEventSynchronize(marks.back().second);
        c->last_stages.clear();
        if (c->trace) fprintf(stderr, "[swb trace] %s:", what);
        for (size_t i = 1; i < marks.size(); i++) {
            float ms = 0;
            cudaEventElapsedTime(&ms, marks[i - 1].second, marks[i].second);
            c->last_stages.emplace_back(marks[i].first, (double)ms);
            if (c->trace) fprintf(stderr, " %s=%.3fms", marks[i].first, ms);
        }
        {
            std::vector<std::pair<const char*, double>> sums;
            for (auto& sp : spans) {
                float ms = 0;
                cudaEventSynchronize(sp.b);
                cudaEventElapsedTime(&ms, sp.a, sp.b);
                bool found = false;
                for (auto& kv : sums)
                    if (kv.first == sp.name) { kv.second += ms; found = true; }
                if (!found) sums.emplace_back(sp.name, (double)ms);
                cudaEventDestroy(sp.a);
                cudaEventDestroy(sp.b);
            }
            for (auto& kv : sums) {
                c->last_stages.emplace_back(kv.first, kv.second);
                if (c->trace) fprintf(stderr, " [%s=%.3fms]", kv.first, kv.second);
            }
        }
        for (auto& kv : counters) c->last_stages.emplace_back(kv.first, (double)*kv.second / 1e6);
        float tot = 0;
        cudaEventElapsedTime(&tot, marks.front().second, marks.back().second);
        c->last_stages.emplace_back("total", (double)tot);
        if (c->trace) fprintf(stderr, " total=%.3fms\n", tot);
        for (auto& m : marks) cudaEventDestroy(m.second);
    }
};

// implemented in ntt.cu
int ntt_build_tables(swb_ctx* c);

}  // namespace swb
