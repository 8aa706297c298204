// Variable-base multi-scalar multiplication over BLS12-377 G1 (Pippenger, bucket method).
//
// Replaces ark_ec::msm::VariableBaseMSM::multi_scalar_mul (ark-ec 0.3 msm/variable_base.rs),
// the hot loop of kzg10::commit / open under Marlin::index and Marlin::prove (reference
// src/marlin/mod.rs:75,92; src/merkle_tree/simple_merkle_tree.rs:83,119).  arkworks uses unsigned
// c-bit windows with 2^c - 1 Jacobian buckets per window and one rayon task per window; here:
//
//   1. k_msm_digits        scalars -> signed c-bit digits (halves the bucket count); one
//                           (bucket, point index | sign) pair per scalar and window, window-major; one
//                           instance per width c, which is a template parameter
//   2. radix_sort_segmented pairs grouped by bucket inside each window (radix_sort.cu)
//   3. k_msm_range_count    the sorted positions are cut into fixed-length ranges; runs per range,
//                           exclusive scan = where each range writes its partial sums
//   4. k_msm_accumulate     one thread per range: XYZZ += +-base (mixed additions), one partial
//                           sum per run of equal bucket ids -- work per thread is bounded whatever
//                           the scalar distribution
//   5. k_msm_gather (+ k_msm_heavy_chunks / k_msm_heavy_finish for buckets with many partial sums)
//                           partial sums of one bucket -> the bucket
//   6. k_msm_segments / k_msm_bit_sums / k_msm_bit_tree / k_msm_bit_final
//                           sum_k k * B_k per bucket set: running sums per segment, then plain sums
//                           selected by the bits of the segment index, reduced as trees
//   7. host                 Horner over the bucket-set sums (c doublings each) and normalisation
//
// With window tables (swb_bases_precompute, fixed_base.cu) digit j of a scalar selects the precomputed
// point 2^(c*j) * P, so all digits share ONE bucket set: steps 2-6 run on a single segment of n * W
// pairs and step 7 has nothing to fold.  msm_begin / msm_end split a call so that the independent MSMs of the
// queue (msm_queue_*, ctx.hpp) overlap on slots with streams and scratch of their own.
//
// The result is the affine value (as a Z = 1 Jacobian), which is unique, hence bit-identical to
// what arkworks' callers see after into_affine().
#include <algorithm>
#include <memory>

#include "msm_common.cuh"

namespace swb {

// 104-byte ABI records -> 96-byte device records; infinity -> (0,0)
__global__ void k_bases_convert(Fq* __restrict__ out, const uint8_t* __restrict__ in, size_t n) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t* src = reinterpret_cast<const uint32_t*>(in + i * 104);
    const bool inf = (src[24] & 0xffu) != 0;
    uint32_t* dst = reinterpret_cast<uint32_t*>(out + 2 * i);
#pragma unroll
    for (int k = 0; k < 24; k++) dst[k] = inf ? 0u : src[k];
}

// ---- host-side tail ------------------------------------------------------------------------
static void xyzz_to_out(const G1Xyzz& p, swb_g1_jacobian* out) {
    memset(out, 0, sizeof *out);
    Fq one = Fq::one();
    if (p.is_identity()) {
        memcpy(out->y.l, one.l, 48);    // (0, 1, 0) = GroupProjective::zero()
        return;
    }
    Fq inv = (p.zz * p.zzz).inverse();          // 1 / (zz * zzz)
    Fq x = p.x * (p.zzz * inv);                 // X / ZZ
    Fq y = p.y * (p.zz * inv);                  // Y / ZZZ
    memcpy(out->x.l, x.l, 48);
    memcpy(out->y.l, y.l, 48);
    memcpy(out->z.l, one.l, 48);
}

static int pick_window(swb_ctx* c, size_t n) {
    if (c->msm_window_override) return c->msm_window_override;
    int lg = 0;
    while (((size_t)1 << lg) < n) lg++;
    // measured on B200 (tools/msm_sweep.py, profiles/r1_msm_window_sweep.json): best signed-window width
    // per log2(n); small sizes are launch-latency bound and flat in c
    static const int best[27] = {4, 4, 4, 4, 4, 5, 6, 7, 8, 8, 8, 9, 11, 11, 11, 11, 11, 11, 15, 15, 15, 16, 17, 18, 19, 19, 20};
    return lg <= 26 ? best[lg] : 20;
}

// streams, event and pinned result buffer of a slot, created on first use
static int slot_prepare(swb_ctx* c, int slot) {
    swb_ctx::MsmSlot& sl = c->msm_slot[slot];
    if (!sl.host_wins) SWB_CUDA(c, cudaMallocHost(&sl.host_wins, sizeof(G1Xyzz) * 2 * MSM_MAX_WINDOWS));
    if (slot > 0 && !sl.work) {
        int lo = 0, hi = 0;
        SWB_CUDA(c, cudaDeviceGetStreamPriorityRange(&lo, &hi));     // hi is the numerically smaller value
        SWB_CUDA(c, cudaStreamCreateWithPriority(&sl.work, cudaStreamNonBlocking, lo));
        SWB_CUDA(c, cudaStreamCreateWithPriority(&sl.tail, cudaStreamNonBlocking, hi));
        SWB_CUDA(c, cudaEventCreateWithFlags(&sl.ev, cudaEventDisableTiming));
    }
    return SWB_OK;
}

static int msm_enqueue(swb_ctx* c, int slot, const swb_bases* bases, const MsmBatch& batch, BucketShard shard, int montgomery);

// The table rule: window tables pay once the buckets hold a few points each (n * W >= 8 * 2^(c-1) per bucket set), unless
// swb_msm_set_table_policy or a window width set with swb_msm_set_window_bits says otherwise.
static bool msm_use_tables(const swb_ctx* c, const swb_bases* b, size_t n, size_t sets) {
    return b->tab_w > 0 && !c->msm_window_override && c->msm_table_policy >= 0 &&
           (c->msm_table_policy > 0 || n * (size_t)b->tab_w >= ((size_t)8 << (b->tab_c - 1)) * sets);
}

// can these vectors run as ONE batched MSM (one bucket set each over the handle's window tables)?
static bool msm_can_batch(swb_ctx* c, const swb_bases* bases, size_t count, const size_t* ns) {
    if (!bases || count < 2 || count > (size_t)MSM_MAX_BATCH) return false;
    size_t total = 0;
    for (size_t k = 0; k < count; k++) total += ns[k];
    return total < ((size_t)1 << 31) && msm_use_tables(c, bases, total, count);
}

void msm_plan_pairs(const swb_ctx* c, MsmPlan& pl) {
    // enough threads to fill the GPU (>= ~512 per SM) but at most 128 additions each
    const size_t want = pl.total / ((size_t)c->sm_count * 512);
    uint32_t len = 16;
    while (len < 128 && len < want) len <<= 1;
    pl.range_len = len;
    pl.nranges = (uint32_t)((pl.total + len - 1) / len);
    // batch-affine pair sums first when buckets are well filled and the input is large enough to amortise the block-wide
    // inversions (swb_msm_set_pair_sums: 0 never, 1 automatic, 1 + k forces k levels)
    int levels = 0;
    if (c->msm_pair_policy >= 2) levels = c->msm_pair_policy - 1;
    else if (c->msm_pair_policy == 1 && pl.total >= MSM_PAIR_MIN_PAIRS) {
        // a level pays while most aligned blocks of 2^L positions still lie inside one bucket
        const double per_bucket = pl.nb ? (double)pl.total / (double)pl.nb : 0.0;
        while (levels < MSM_PAIR_MAX_LEVELS && per_bucket >= (double)(8u << levels)) levels++;
    }
    pl.pair_levels = pl.total >= 2 ? levels : 0;
}

// Every decision of one MSM, from the context's settings, the bases, the batch and the bucket shard.  Under compaction
// the number of pairs is known only after the digits kernel: the sizes planned here are then upper bounds for the
// scratch, and msm_launch_digits_sort plans the ranges and pair sums again.
static int msm_plan(swb_ctx* c, const swb_bases* bases, const MsmBatch& batch, BucketShard shard, MsmPlan& pl) {
    pl = MsmPlan{};
    pl.n = batch.start[batch.count];
    const bool tables = batch.count > 1 || msm_use_tables(c, bases, pl.n, 1);    // a batch always runs over tables
    pl.cb = tables ? bases->tab_c : pick_window(c, pl.n);
    pl.ndig = tables ? bases->tab_w : (254 + pl.cb - 1) / pl.cb;
    pl.nwin = tables ? (int)batch.count : pl.ndig;        // bucket sets
    SWB_REQUIRE(c, pl.ndig <= MSM_MAX_WINDOWS, "msm: too many windows");
    pl.tab_stride = tables ? bases->n : 0;
    pl.B = 1u << (pl.cb - 1);
    if (shard.world > 1 && (uint32_t)shard.world <= pl.B / 2) {
        // bucket sharding: this rank fills the buckets b = rank (mod world) of every set.  On the table path (one
        // set, pair order free) the other ranks' pairs are dropped right in the digits kernel.
        while ((1 << pl.shard_shift) < shard.world) pl.shard_shift++;
        pl.B >>= pl.shard_shift;
        pl.shard_rank = (uint32_t)shard.rank;
        pl.compact = tables;
    } else if (shard.world > 1 && shard.rank != 0) {
        pl.idle = true;           // too few buckets to split (tiny MSM, narrow window)
        return SWB_OK;
    }
    pl.nb = (uint32_t)pl.nwin * pl.B;
    pl.key_space = tables ? pl.nb : pl.B;     // table path: one segment, the key says which set; plain path: a segment per set
    pl.total = pl.n * (size_t)pl.ndig;
    pl.seg_len = tables ? pl.total : pl.n;
    SWB_REQUIRE(c, pl.total < ((size_t)1 << 32), "msm: n * windows must be < 2^32");
    msm_plan_pairs(c, pl);
    if (pl.compact) {       // whatever number of pairs survives: at most this many ranges
        const size_t a = pl.total / 128 + 1, b = (size_t)c->sm_count * 512 + 1;
        pl.nranges = (uint32_t)(a > b ? a : b);
    }
    pl.pcap = pl.nranges + pl.nb;
    return SWB_OK;
}

// the checks of one request, made by the single calls and at submission to the queue
static int msm_check(swb_ctx* c, const swb_bases* bases, size_t offset, const void* scalars_dev, size_t n) {
    SWB_REQUIRE(c, bases != nullptr, "msm: bad batch");
    SWB_REQUIRE(c, bases->ctx == c, "msm: bases belong to another context");
    SWB_REQUIRE(c, offset <= bases->n && n <= bases->n - offset, "msm: offset + n exceeds the loaded bases");
    SWB_REQUIRE(c, n == 0 || scalars_dev != nullptr, "msm: NULL scalars");
    SWB_REQUIRE(c, n < ((size_t)1 << 31), "msm: n must be < 2^31");
    return SWB_OK;
}

// One MSM split in two: msm_begin enqueues everything up to the device->host copy of the bucket-set sums (slot 0: on the
// context's stream; slot > 0: on the slot's own streams, after the work already queued on the context's stream), msm_end
// waits for it and finishes on the host.  A slot holds one MSM at a time.  msm_begin_batch runs several scalar vectors
// over one handle with window tables as ONE pipeline (a bucket set per vector, see msm_can_batch); msm_end then
// delivers `count` results.  Every vector has passed msm_check.
static int msm_begin_batch(swb_ctx* c, int slot, const swb_bases* bases, size_t count, const size_t* offsets, const void* const* scalars_dev,
                           const size_t* ns, int montgomery, BucketShard shard) {
    SWB_REQUIRE(c, slot >= 0 && slot < swb_ctx::MSM_SLOTS, "msm: bad slot");
    SWB_REQUIRE(c, !c->msm_slot[slot].active, "msm: slot already holds an MSM");
    SWB_REQUIRE(c, count >= 1 && count <= (size_t)MSM_MAX_BATCH, "msm: bad batch");
    MsmBatch batch{};
    size_t total = 0;
    uint32_t kept = 0;
    for (size_t k = 0; k < count; k++) {
        // empty vectors keep their bucket set (it stays empty), so that results stay in the caller's order
        batch.scalars[kept] = (const uint32_t*)scalars_dev[k];
        batch.start[kept] = (uint32_t)total;
        batch.offset[kept] = (uint32_t)offsets[k];
        total += ns[k];
        kept++;
    }
    SWB_REQUIRE(c, total < ((size_t)1 << 31), "msm: n must be < 2^31");
    batch.start[kept] = (uint32_t)total;
    batch.count = kept;
    SWB_REQUIRE(c, count == 1 || msm_can_batch(c, bases, count, ns) || total == 0, "msm: these vectors cannot run as one batch");
    SWB_CUDA(c, cudaSetDevice(c->device));
    int rc = slot_prepare(c, slot);
    if (rc != SWB_OK) return rc;
    swb_ctx::MsmSlot& sl = c->msm_slot[slot];
    const size_t n = total;
    sl.empty = n == 0;
    sl.nres = (int)count;
    if (n == 0) {
        sl.active = true;
        return SWB_OK;
    }
    cudaStream_t main_stream = c->stream;
    if (slot > 0) {
        // inputs (scalars, bases) are produced on the context's stream: the slot starts after them
        SWB_CUDA(c, cudaEventRecord(sl.ev, main_stream));
        SWB_CUDA(c, cudaStreamWaitEvent(sl.work, sl.ev, 0));
        c->stream = sl.work;
        c->scratch_slot = slot;
    }
    rc = msm_enqueue(c, slot, bases, batch, shard, montgomery);
    c->stream = main_stream;
    c->scratch_slot = 0;
    if (rc == SWB_OK) sl.active = true;
    return rc;
}

static int msm_begin(swb_ctx* c, int slot, const swb_bases* bases, size_t offset, const void* scalars_dev, size_t n, int montgomery,
                     BucketShard shard) {
    return msm_begin_batch(c, slot, bases, 1, &offset, &scalars_dev, &n, montgomery, shard);
}

// outs: one result per vector of the batch (one for a plain msm_begin)
static int msm_end(swb_ctx* c, int slot, swb_g1_jacobian* out) {
    SWB_REQUIRE(c, slot >= 0 && slot < swb_ctx::MSM_SLOTS && out, "msm: bad slot");
    swb_ctx::MsmSlot& sl = c->msm_slot[slot];
    SWB_REQUIRE(c, sl.active, "msm: slot holds no MSM");
    sl.active = false;
    if (sl.empty) {
        for (int k = 0; k < sl.nres; k++) xyzz_to_out(G1Xyzz::identity(), out + k);
        return SWB_OK;
    }
    SWB_CUDA(c, cudaSetDevice(c->device));
    SWB_CUDA(c, cudaStreamSynchronize(slot > 0 ? sl.tail : c->stream));
    const G1Xyzz* hw = static_cast<const G1Xyzz*>(sl.host_wins);
    // a bucket shard holds R = sum_k (k + 1) B_k over its LOCAL bucket numbers k; the global number of local bucket k
    // is world * k + rank, so its share of the set's sum is
    //     sum_k (world * k + rank + 1) B_k = world * R - (world - rank - 1) * S,   S = plain sum (second half of the buffer)
    auto small_mul = [](const G1Xyzz& p, uint32_t k) {
        G1Xyzz t = G1Xyzz::identity();
        for (int b = 31; b >= 0; b--) {
            t = t.dbl();
            if ((k >> b) & 1u) t.add(p);
        }
        return t;
    };
    auto set_sum = [&](int w) {
        G1Xyzz r = hw[w];
        if (sl.shard_world > 1) {
            r = small_mul(r, (uint32_t)sl.shard_world);
            G1Xyzz t = small_mul(hw[sl.nwin + w], (uint32_t)(sl.shard_world - sl.shard_rank - 1));
            t.y = t.y.neg();
            r.add(t);
        }
        return r;
    };
    if (sl.batched) {                       // one bucket set per vector: its sum is the vector's result
        for (int k = 0; k < sl.nres; k++) xyzz_to_out(set_sum(k), out + k);
        return SWB_OK;
    }
    // Horner over the bucket sets, most significant first
    G1Xyzz acc = set_sum(sl.nwin - 1);
    for (int w = sl.nwin - 2; w >= 0; w--) {
        for (int k = 0; k < sl.cb; k++) acc = acc.dbl();
        acc.add(set_sum(w));
    }
    xyzz_to_out(acc, out);
    return SWB_OK;
}

// the bucket shard of swb_msm_set_bucket_shard, under which the swb_msm_* entry points run
static BucketShard ctx_bucket_shard(const swb_ctx* c) { return {c->bucket_rank, c->bucket_world}; }

static int msm_run(swb_ctx* c, const swb_bases* bases, size_t offset, const void* scalars_dev, size_t n, int montgomery,
                   swb_g1_jacobian* out) {
    SWB_REQUIRE(c, out != nullptr, "msm: NULL argument");
    int rc = msm_check(c, bases, offset, scalars_dev, n);
    if (rc == SWB_OK) rc = msm_begin(c, 0, bases, offset, scalars_dev, n, montgomery, ctx_bucket_shard(c));
    if (rc != SWB_OK) return rc;
    return msm_end(c, 0, out);
}

// scalars in host memory (32 bytes each): copied to device scratch first
static int msm_run_host(swb_ctx* c, const swb_bases* bases, size_t offset, const void* scalars_host, size_t n, int montgomery,
                        swb_g1_jacobian* out) {
    SWB_REQUIRE(c, n == 0 || scalars_host != nullptr, "msm: NULL scalars");
    void* d = nullptr;
    if (n) {
        SWB_CUDA(c, cudaSetDevice(c->device));
        d = get_scratch(c, "msm_scalars", n * 32);
        if (!d) return SWB_ENOMEM;
        SWB_CUDA(c, cudaMemcpyAsync(d, scalars_host, n * 32, cudaMemcpyHostToDevice, c->stream));
    }
    return msm_run(c, bases, offset, d, n, montgomery, out);
}

// ---- the MSM queue (ctx.hpp) ----------------------------------------------------------------------

int msm_queue_submit(swb_ctx* c, const swb_bases* bases, size_t offset, const void* scalars_dev, size_t n, int montgomery,
                     BucketShard shard, size_t* id) {
    const int rc = msm_check(c, bases, offset, scalars_dev, n);
    if (rc != SWB_OK) return rc;
    *id = c->msm_queue_next++;
    c->msm_queue.emplace(*id, swb_ctx::MsmRequest{bases, offset, n, scalars_dev, montgomery, shard});
    return SWB_OK;
}

// finishes the MSM running on slot s, if there is one, and hands its results to the requests it serves (a batch on slot
// 0 serves several, in submission order)
static int msm_queue_collect(swb_ctx* c, int s) {
    if (!c->msm_slot[s].active) return SWB_OK;
    swb_g1_jacobian outs[MSM_MAX_BATCH];
    const int rc = msm_end(c, s, outs);
    int k = 0;
    for (auto& kv : c->msm_queue) {
        swb_ctx::MsmRequest& r = kv.second;
        if (r.slot != s || r.done) continue;
        r.out = outs[k++];
        r.done = rc == SWB_OK;
    }
    return rc;
}

int msm_queue_launch(swb_ctx* c, bool* launched) {
    *launched = false;
    auto it = c->msm_queue.begin();
    while (it != c->msm_queue.end() && it->second.slot >= 0) ++it;
    if (it == c->msm_queue.end()) return SWB_OK;
    *launched = true;
    swb_ctx::MsmRequest& first = it->second;
    if (!first.single) {
        swb_ctx::MsmRequest* run[MSM_MAX_BATCH];
        size_t offs[MSM_MAX_BATCH], ns[MSM_MAX_BATCH];
        const void* scs[MSM_MAX_BATCH];
        size_t cnt = 0;
        for (; it != c->msm_queue.end() && cnt < (size_t)MSM_MAX_BATCH; ++it, ++cnt) {
            swb_ctx::MsmRequest& r = it->second;
            if (r.slot >= 0 || r.bases != first.bases || r.montgomery != first.montgomery || r.shard.rank != first.shard.rank ||
                r.shard.world != first.shard.world)
                break;
            run[cnt] = &r;
            offs[cnt] = r.offset; ns[cnt] = r.n; scs[cnt] = r.scalars;
        }
        if (cnt >= 2 && msm_can_batch(c, first.bases, cnt, ns)) {
            // the batch runs on the context's stream with slot 0's scratch: the other slots and the previous batch finish
            // first.  Its results are collected when one of them is asked for.
            int rc = SWB_OK;
            for (int s = 0; s < swb_ctx::MSM_SLOTS && rc == SWB_OK; s++) rc = msm_queue_collect(c, s);
            if (rc == SWB_OK) rc = msm_begin_batch(c, 0, first.bases, cnt, offs, scs, ns, first.montgomery, first.shard);
            if (rc != SWB_OK) return rc;
            for (size_t k = 0; k < cnt; k++) run[k]->slot = 0;
            return SWB_OK;
        }
        for (size_t k = 0; k < cnt; k++) run[k]->single = true;      // this run goes out one request at a time
    }
    const int s = c->msm_next_slot;
    c->msm_next_slot = s == 1 ? 2 : 1;
    int rc = msm_queue_collect(c, s);
    if (rc == SWB_OK) rc = msm_begin(c, s, first.bases, first.offset, first.scalars, first.n, first.montgomery, first.shard);
    if (rc != SWB_OK) return rc;
    first.slot = s;
    return SWB_OK;
}

int msm_queue_flush(swb_ctx* c) {
    for (bool launched = true; launched;) {
        const int rc = msm_queue_launch(c, &launched);
        if (rc != SWB_OK) return rc;
    }
    return SWB_OK;
}

int msm_queue_result(swb_ctx* c, size_t id, swb_g1_jacobian* out) {
    auto it = c->msm_queue.find(id);
    SWB_REQUIRE(c, out != nullptr && it != c->msm_queue.end(), "msm queue: no such request (its result was taken, or the queue abandoned)");
    int rc = it->second.slot < 0 ? msm_queue_flush(c) : SWB_OK;
    if (rc == SWB_OK && !it->second.done) rc = msm_queue_collect(c, it->second.slot);
    if (rc != SWB_OK) return rc;
    *out = it->second.out;
    c->msm_queue.erase(it);
    return SWB_OK;
}

int msm_queue_drain(swb_ctx* c) {
    int rc = msm_queue_flush(c);
    for (int s = 0; s < swb_ctx::MSM_SLOTS && rc == SWB_OK; s++) rc = msm_queue_collect(c, s);
    return rc;
}

void msm_queue_abandon(swb_ctx* c) {
    const std::string err = c->err;         // the failure that led here stays the context's last error
    swb_g1_jacobian dummy[MSM_MAX_BATCH];                       // slot 0 may hold a batch
    for (int s = 0; s < swb_ctx::MSM_SLOTS; s++)
        if (c->msm_slot[s].active) msm_end(c, s, dummy);        // waits for the slot's work
    c->msm_queue.clear();
    c->err = err;
}

static int msm_enqueue(swb_ctx* c, int slot, const swb_bases* bases, const MsmBatch& batch, BucketShard shard, int montgomery) {
    swb_ctx::MsmSlot& sl = c->msm_slot[slot];
    MsmPlan pl;
    int rc = msm_plan(c, bases, batch, shard, pl);
    if (rc != SWB_OK) return rc;
    if (pl.idle) {
        sl.empty = true;
        return SWB_OK;
    }
    MsmBuffers bf{};
    bf.keys = (uint32_t*)get_scratch(c, "msm_keys", msm_alt_offset(pl.total) * 4 * 2);
    bf.vals = (uint32_t*)get_scratch(c, "msm_vals", msm_alt_offset(pl.total) * 4 * 2);
    bf.range_off = (uint32_t*)get_scratch(c, "msm_roff", ((size_t)pl.nranges + 2) * 4);
    bf.pkey = (uint32_t*)get_scratch(c, "msm_pkey", (size_t)pl.pcap * 4);
    bf.pstart = (uint32_t*)get_scratch(c, "msm_pstart", ((size_t)pl.nb + 2) * 4);
    bf.heavy = (uint32_t*)get_scratch(c, "msm_heavy", ((size_t)pl.nb + 2) * 4);
    bf.partial = (G1Xyzz*)get_scratch(c, "msm_partial", (size_t)pl.pcap * sizeof(G1Xyzz));
    bf.buckets = (G1Xyzz*)get_scratch(c, "msm_buckets", (size_t)pl.nb * sizeof(G1Xyzz));
    {
        const size_t segs = (size_t)pl.nwin * (pl.B / msm_reduce_seg_len((uint32_t)pl.nwin, pl.B));
        bf.seg = (G1Xyzz*)get_scratch(c, "msm_seg", (2 * segs + 2) * sizeof(G1Xyzz));
        bf.seg2 = (G1Xyzz*)get_scratch(c, "msm_seg2", ((size_t)pl.nwin * 24 * 33 + 2) * sizeof(G1Xyzz));   // [sets][jobs][blocks + 1]
    }
    bf.wins = (G1Xyzz*)get_scratch(c, "msm_wins", (size_t)2 * MSM_MAX_WINDOWS * sizeof(G1Xyzz));
    bf.count = (uint32_t*)get_scratch(c, "msm_count", 64);
    if (!bf.count || !bf.keys || !bf.vals || !bf.range_off || !bf.pkey || !bf.pstart || !bf.heavy || !bf.partial ||
        !bf.buckets || !bf.seg || !bf.seg2 || !bf.wins)
        return SWB_ENOMEM;
    const uint32_t *sorted_keys = nullptr, *sorted_vals = nullptr;
    std::unique_ptr<StageTimer> tmp(slot == 0 ? new StageTimer(c, "msm") : nullptr);   // stage timing: slot 0 only
    struct { StageTimer* t; void mark(const char* n) { if (t) t->mark(n); } } tm{tmp.get()};
    rc = msm_launch_digits_sort(c, pl, bf, batch, montgomery, &sorted_keys, &sorted_vals, tmp.get());
    if (rc != SWB_OK) return rc;
    tm.mark("count");
    if (pl.pair_levels > 0) {
        static const char* const tags[MSM_PAIR_MAX_LEVELS + 1] = {"", "msm_pair_r1", "msm_pair_r2", "msm_pair_r3", "msm_pair_r4"};
        for (int l = 1; l <= pl.pair_levels; l++) {
            const size_t slots = (pl.total + ((size_t)1 << l) - 1) >> l;
            bf.pair_sums[l] = (Fq*)get_scratch(c, tags[l], slots * 2 * sizeof(Fq) + 64);
            if (!bf.pair_sums[l]) return SWB_ENOMEM;
        }
        bf.pair_lvl = (uint8_t*)get_scratch(c, "msm_pair_lvl", (pl.total + 1) / 2 + 64);
        if (!bf.pair_lvl) return SWB_ENOMEM;
        rc = msm_launch_pair_sums(c, pl, bf.pair_sums, bf.pair_lvl, pl.pair_levels, sorted_keys, sorted_vals, bases->xy, tmp.get());
        if (rc != SWB_OK) return rc;
        tm.mark("pair_sums");
    }
    rc = msm_launch_accumulate(c, pl, bf, sorted_keys, sorted_vals, bases->xy);
    if (rc != SWB_OK) return rc;
    tm.mark("accumulate");
    if (slot > 0) {
        // the bucket tail is latency-bound and small: on the slot's high-priority stream its blocks get
        // the SM slots that another MSM's accumulation frees, instead of queueing behind it
        SWB_CUDA(c, cudaEventRecord(sl.ev, sl.work));
        SWB_CUDA(c, cudaStreamWaitEvent(sl.tail, sl.ev, 0));
        c->stream = sl.tail;
    }
    rc = msm_launch_gather(c, pl, bf);
    if (rc != SWB_OK) return rc;
    tm.mark("gather");
    rc = msm_launch_reduce(c, pl, bf);
    if (rc != SWB_OK) return rc;
    tm.mark("reduce");
    if (c->trace > 1) {   // SWB_TRACE=2: partial-sum statistics
        uint32_t np = 0, nheavy = 0;
        cudaMemcpyAsync(&np, bf.range_off + pl.nranges, 4, cudaMemcpyDeviceToHost, c->stream);
        cudaMemcpyAsync(&nheavy, bf.heavy, 4, cudaMemcpyDeviceToHost, c->stream);
        cudaStreamSynchronize(c->stream);
        fprintf(stderr, "[swb trace] msm: n=%zu c=%d windows=%d buckets=%u range_len=%u ranges=%u partials=%u heavy_buckets=%u\n", pl.n,
                pl.cb, pl.nwin, pl.nb, pl.range_len, pl.nranges, np, nheavy);
    }

    sl.nwin = pl.nwin;
    sl.cb = pl.cb;
    sl.batched = batch.count > 1;
    sl.shard_rank = (int)pl.shard_rank;
    sl.shard_world = 1 << pl.shard_shift;
    SWB_CUDA(c, cudaMemcpyAsync(sl.host_wins, bf.wins, sizeof(G1Xyzz) * pl.nwin, cudaMemcpyDeviceToHost, c->stream));
    if (pl.shard_shift)
        SWB_CUDA(c, cudaMemcpyAsync(static_cast<G1Xyzz*>(sl.host_wins) + pl.nwin, bf.wins + MSM_MAX_WINDOWS, sizeof(G1Xyzz) * pl.nwin,
                                    cudaMemcpyDeviceToHost, c->stream));
    return SWB_OK;
}

}  // namespace swb

using namespace swb;

extern "C" {

int swb_bases_load_dev(swb_ctx* c, const swb_g1_affine* dev, size_t n, swb_bases** out) {
    if (!c) return SWB_EARG;
    SWB_REQUIRE(c, out != nullptr, "bases_load: out is NULL");
    SWB_REQUIRE(c, n == 0 || dev != nullptr, "bases_load: NULL points");
    SWB_CUDA(c, cudaSetDevice(c->device));
    swb_bases* b = new swb_bases();
    b->ctx = c;
    b->n = n;
    cudaError_t e = cudaMalloc(&b->xy, (n ? n : 1) * 96);
    if (e != cudaSuccess) {
        delete b;
        return set_err(c, SWB_ENOMEM, "bases_load: cudaMalloc(%zu) failed: %s", n * 96, cudaGetErrorString(e));
    }
    if (n) {
        k_bases_convert<<<(unsigned)((n + 255) / 256), 256, 0, c->stream>>>(b->xy, (const uint8_t*)dev, n);
        c->launches++;
        e = cudaGetLastError();
        if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
        if (e != cudaSuccess) {
            cudaFree(b->xy);
            delete b;
            return cuda_fail(c, e, "k_bases_convert");
        }
    }
    *out = b;
    return SWB_OK;
}

int swb_bases_load(swb_ctx* c, const swb_g1_affine* host, size_t n, swb_bases** out) {
    if (!c) return SWB_EARG;
    SWB_REQUIRE(c, out != nullptr, "bases_load: out is NULL");
    SWB_REQUIRE(c, n == 0 || host != nullptr, "bases_load: NULL points");
    SWB_CUDA(c, cudaSetDevice(c->device));
    void* staging = nullptr;
    if (n) {
        cudaError_t e = cudaMalloc(&staging, n * sizeof(swb_g1_affine));
        if (e != cudaSuccess) return set_err(c, SWB_ENOMEM, "bases_load: staging cudaMalloc failed: %s", cudaGetErrorString(e));
        e = cudaMemcpyAsync(staging, host, n * sizeof(swb_g1_affine), cudaMemcpyHostToDevice, c->stream);
        if (e != cudaSuccess) {
            cudaFree(staging);
            return cuda_fail(c, e, "bases_load H2D");
        }
    }
    int rc = swb_bases_load_dev(c, (const swb_g1_affine*)staging, n, out);
    if (staging) cudaFree(staging);
    return rc;
}

size_t swb_bases_len(const swb_bases* b) { return b ? b->n : 0; }

void swb_bases_free(swb_bases* b) {
    if (!b) return;
    if (b->ctx) sync_all_streams(b->ctx);
    if (b->xy) cudaFree(b->xy);
    delete b;
}

int swb_msm_plan(swb_ctx* c, size_t n, int* window_bits, int* windows) {
    if (!c) return SWB_EARG;
    const int cb = pick_window(c, n ? n : 1);
    if (window_bits) *window_bits = cb;
    if (windows) *windows = (254 + cb - 1) / cb;
    return SWB_OK;
}

int swb_set_msm_shard(swb_ctx* c, int rank, int world, swb_combine_fn combine, void* user) {
    if (!c) return SWB_EARG;
    if (world <= 1) {
        c->shard_rank = 0; c->shard_world = 1; c->shard_combine = nullptr; c->shard_user = nullptr;
        return SWB_OK;
    }
    SWB_REQUIRE(c, rank >= 0 && rank < world, "set_msm_shard: rank out of range");
    SWB_REQUIRE(c, c->msm_peers.empty() && c->msm_primaries.empty(), "set_msm_shard: the context shares its MSMs with peer contexts (swb_set_msm_peers)");
    // without a callback the partial results travel through the context's own communicator (swb_comm_init)
    SWB_REQUIRE(c, combine || (c->comm && c->comm_world == world && c->comm_rank == rank),
                "set_msm_shard: no combine callback and no communicator of this shape (swb_comm_init)");
    c->shard_rank = rank; c->shard_world = world; c->shard_combine = combine; c->shard_user = user;
    return SWB_OK;
}

int swb_set_msm_peers(swb_ctx* c, swb_ctx* const* peers, int n_peers) {
    if (!c) return SWB_EARG;
    SWB_REQUIRE(c, n_peers >= 0 && n_peers < 1024 && (n_peers == 0 || peers), "set_msm_peers: bad peer list");
    auto idle = [](const swb_ctx* x) {
        for (auto& sl : x->msm_slot)
            if (sl.active) return false;
        return x->msm_queue.empty();
    };
    SWB_REQUIRE(c, idle(c), "set_msm_peers: an MSM is in flight");
    for (swb_ctx* p : c->msm_peers) SWB_REQUIRE(c, idle(p), "set_msm_peers: an MSM is in flight on a peer");
    if (n_peers > 0) {
        SWB_REQUIRE(c, c->shard_world <= 1, "set_msm_peers: the context shards through swb_set_msm_shard");
        SWB_REQUIRE(c, c->msm_primaries.empty(), "set_msm_peers: the context is a peer of another context");
    }
    for (int i = 0; i < n_peers; i++) {
        const swb_ctx* p = peers[i];
        SWB_REQUIRE(c, p != nullptr, "set_msm_peers: NULL peer");
        SWB_REQUIRE(c, p != c, "set_msm_peers: a context cannot be its own peer");
        for (int j = 0; j < i; j++) SWB_REQUIRE(c, peers[j] != p, "set_msm_peers: repeated peer");
        SWB_REQUIRE(c, p->msm_peers.empty() && p->shard_world <= 1, "set_msm_peers: a peer has peers or a shard of its own");
        SWB_REQUIRE(c, idle(p), "set_msm_peers: an MSM is in flight on a peer");
    }
    if (n_peers > 0 && !c->peer_ev) {
        SWB_CUDA(c, cudaSetDevice(c->device));
        SWB_CUDA(c, cudaEventCreateWithFlags(&c->peer_ev, cudaEventDisableTiming));
    }
    // direct access between the devices where they allow it; elsewhere cudaMemcpyPeerAsync stages through the host
    for (int i = 0; i < n_peers; i++) {
        const int a = c->device, b = peers[i]->device;
        int ab = 0, ba = 0;
        if (a == b || cudaDeviceCanAccessPeer(&ab, a, b) != cudaSuccess || cudaDeviceCanAccessPeer(&ba, b, a) != cudaSuccess) continue;
        if (ab && cudaSetDevice(a) == cudaSuccess) cudaDeviceEnablePeerAccess(b, 0);
        if (ba && cudaSetDevice(b) == cudaSuccess) cudaDeviceEnablePeerAccess(a, 0);
        cudaGetLastError();              // cudaErrorPeerAccessAlreadyEnabled, or access refused: the copies are staged
    }
    cudaSetDevice(c->device);
    for (swb_ctx* p : c->msm_peers) p->msm_primaries.erase(std::find(p->msm_primaries.begin(), p->msm_primaries.end(), c));
    c->msm_peers.assign(peers, peers + n_peers);
    for (swb_ctx* p : c->msm_peers) p->msm_primaries.push_back(c);
    return SWB_OK;
}

uint64_t swb_peer_copy_bytes(const swb_ctx* c) { return c ? c->peer_bytes : 0; }

int swb_msm_set_bucket_shard(swb_ctx* c, int rank, int world) {
    if (!c) return SWB_EARG;
    if (world <= 1) { c->bucket_rank = 0; c->bucket_world = 1; return SWB_OK; }
    SWB_REQUIRE(c, (world & (world - 1)) == 0 && world <= 1024, "msm_set_bucket_shard: world must be a power of two <= 1024");
    SWB_REQUIRE(c, rank >= 0 && rank < world, "msm_set_bucket_shard: rank out of range");
    c->bucket_rank = rank;
    c->bucket_world = world;
    return SWB_OK;
}

int swb_msm_set_pair_sums(swb_ctx* c, int policy) {
    if (!c) return SWB_EARG;
    SWB_REQUIRE(c, policy >= 0 && policy <= 1 + MSM_PAIR_MAX_LEVELS, "msm_set_pair_sums: 0 (never), 1 (automatic) or 1 + the number of levels (2..5)");
    c->msm_pair_policy = policy;
    return SWB_OK;
}

int swb_msm_set_window_bits(swb_ctx* c, int cb) {
    if (!c) return SWB_EARG;
    SWB_REQUIRE(c, cb == 0 || (cb >= 2 && cb <= 24), "msm_set_window_bits: c must be 0 or in [2,24]");
    c->msm_window_override = cb;
    return SWB_OK;
}

int swb_msm_set_table_policy(swb_ctx* c, int policy) {
    if (!c) return SWB_EARG;
    SWB_REQUIRE(c, policy >= -1 && policy <= 1, "msm_set_table_policy: -1 (never), 0 (automatic) or 1 (always)");
    c->msm_table_policy = policy;
    return SWB_OK;
}

int swb_msm_g1_dev(swb_ctx* c, const swb_bases* b, size_t offset, const swb_bigint256* scalars_dev, size_t n,
                   swb_g1_jacobian* out) {
    if (!c) return SWB_EARG;
    return msm_run(c, b, offset, scalars_dev, n, 0, out);
}

int swb_msm_g1_fr_dev(swb_ctx* c, const swb_bases* b, size_t offset, const swb_fr* scalars_dev, size_t n,
                      swb_g1_jacobian* out) {
    if (!c) return SWB_EARG;
    return msm_run(c, b, offset, scalars_dev, n, 1, out);
}

int swb_msm_g1_batch_dev(swb_ctx* c, const swb_bases* b, const size_t* offsets, const void* const* scalars_dev, const size_t* ns,
                         size_t n_msms, int montgomery, swb_g1_jacobian* outs) {
    if (!c) return SWB_EARG;
    SWB_REQUIRE(c, n_msms == 0 || (offsets && scalars_dev && ns && outs), "msm_batch: NULL argument");
    std::vector<size_t> ids(n_msms);
    int rc = SWB_OK;
    for (size_t i = 0; i < n_msms && rc == SWB_OK; i++)
        rc = msm_queue_submit(c, b, offsets[i], scalars_dev[i], ns[i], montgomery, ctx_bucket_shard(c), &ids[i]);
    for (size_t i = 0; i < n_msms && rc == SWB_OK; i++) rc = msm_queue_result(c, ids[i], &outs[i]);
    if (rc != SWB_OK) msm_queue_abandon(c);
    return rc;
}

int swb_msm_g1(swb_ctx* c, const swb_bases* b, size_t offset, const swb_bigint256* scalars_host, size_t n,
               swb_g1_jacobian* out) {
    if (!c) return SWB_EARG;
    return msm_run_host(c, b, offset, scalars_host, n, 0, out);
}

int swb_msm_g1_fr(swb_ctx* c, const swb_bases* b, size_t offset, const swb_fr* scalars_host, size_t n, swb_g1_jacobian* out) {
    if (!c) return SWB_EARG;
    return msm_run_host(c, b, offset, scalars_host, n, 1, out);
}

int swb_g1_sum_jacobian(swb_ctx* c, const swb_g1_jacobian* pts, size_t n, swb_g1_jacobian* out) {
    // pure host arithmetic: the context is only used for error text and may be NULL
    if (!(out && (n == 0 || pts))) return set_err(c, SWB_EARG, "%s", "g1_sum: NULL argument");
    G1Xyzz acc = G1Xyzz::identity();
    for (size_t i = 0; i < n; i++) {
        G1Xyzz p;
        Fq z;
        memcpy(p.x.l, pts[i].x.l, 48);
        memcpy(p.y.l, pts[i].y.l, 48);
        memcpy(z.l, pts[i].z.l, 48);
        if (z.is_zero()) continue;
        p.zz = z.sqr();                 // Jacobian (X, Y, Z) == XYZZ (X, Y, Z^2, Z^3)
        p.zzz = p.zz * z;
        acc.add(p);
    }
    xyzz_to_out(acc, out);
    return SWB_OK;
}

}  // extern "C"
