// Protocol-level C ABI: simpleworks::marlin's surface (reference src/marlin/mod.rs:33-94) on the
// CUDA engine.  Host orchestration (transcript, AHP rounds, KZG bookkeeping) is marlin/marlin.hpp;
// every NTT, MSM and fixed-base table goes to the kernels of this library -- there is no CPU
// engine in libswb200.
#include "ctx.hpp"
#include "marlin/c_api_impl.hpp"
#include "index_ops.hpp"
#include "marlin_ops.hpp"
#include "polyops.hpp"

using namespace swb;
using namespace swb::marlin;

namespace {

// Fr vector in HBM, owned; blocks come from the context's stream-ordered cache (ctx.hpp: vec_alloc)
struct DVec {
    swb_ctx* c = nullptr;
    Fr* p = nullptr;
    size_t n = 0, cap = 0;       // elements in use / elements the block holds
    size_t blk = 0;              // block size in bytes, for vec_free
    DVec() {}
    DVec(const DVec&) = delete;
    DVec& operator=(const DVec&) = delete;
    DVec(DVec&& o) noexcept : c(o.c), p(o.p), n(o.n), cap(o.cap), blk(o.blk) { o.p = nullptr; o.n = o.cap = o.blk = 0; }
    DVec& operator=(DVec&& o) noexcept {
        if (this != &o) {
            release();
            c = o.c; p = o.p; n = o.n; cap = o.cap; blk = o.blk;
            o.p = nullptr; o.n = o.cap = o.blk = 0;
        }
        return *this;
    }
    ~DVec() { release(); }
    void release() {
        if (p && c) vec_free(c, p, blk);
        p = nullptr;
        n = cap = blk = 0;
    }
    size_t size() const { return n; }
};

struct GpuEngine;
// SWB_TRACE=2: every engine operation is bracketed by stream synchronisations and accounted under
// "op:<name>" in the host profile (serialises the stream; for attribution only)
struct OpTimer {
    swb_ctx* c;
    const char* name;
    bool on;
    std::chrono::steady_clock::time_point t0;
    OpTimer(swb_ctx* ctx, const char* n) : c(ctx), name(n), on(ctx->trace >= 2) {
        if (on) { cudaStreamSynchronize(c->stream); t0 = std::chrono::steady_clock::now(); }
    }
    ~OpTimer() {
        if (!on) return;
        cudaStreamSynchronize(c->stream);
        host_profile().acc[std::string("op:") + name] += std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
    }
};

struct GpuEngine {
    using Vec = DVec;
    swb_ctx* c;
    explicit GpuEngine(swb_ctx* ctx) : c(ctx) { cudaSetDevice(c->device); }
    [[noreturn]] void fail(const char* what) { throw MarlinError(std::string(what) + ": " + swb_last_error(c)); }
    void ck(int rc, const char* what) { if (rc != SWB_OK) fail(what); }
    void cu(cudaError_t e, const char* what) {
        if (e != cudaSuccess) throw MarlinError(std::string(what) + ": " + cudaGetErrorString(e));
    }
    // ---- storage ----------------------------------------------------------------------------
    Vec alloc(size_t n) {
        Vec v;
        v.c = c;
        if (!n) return v;
        v.p = static_cast<Fr*>(vec_alloc(c, n * sizeof(Fr), &v.blk));
        if (!v.p) fail("vec_alloc");
        v.n = n;
        v.cap = v.blk / sizeof(Fr);
        return v;
    }
    Vec vzeros(size_t n) {
        OpTimer ot_(c, "vzeros");
        Vec v = alloc(n);
        if (n) cu(cudaMemsetAsync(v.p, 0, n * sizeof(Fr), c->stream), "memset");
        return v;
    }
    Vec vfrom(const std::vector<Fr>& h) {
        OpTimer ot_(c, "vfrom");
        Vec v = alloc(h.size());
        if (!h.empty()) {
            cu(cudaMemcpyAsync(v.p, h.data(), h.size() * sizeof(Fr), cudaMemcpyHostToDevice, c->stream), "H2D");
            cu(cudaStreamSynchronize(c->stream), "sync");     // h may be a temporary
        }
        return v;
    }
    Vec vfrom_ptr(const Fr* h, size_t n) {
        OpTimer ot_(c, "vfrom");
        Vec v = alloc(n);
        if (n) {
            cu(cudaMemcpyAsync(v.p, h, n * sizeof(Fr), cudaMemcpyHostToDevice, c->stream), "H2D");
            cu(cudaStreamSynchronize(c->stream), "sync");     // the caller may free h
        }
        return v;
    }
    void vwrite(Vec& v, size_t at, const Fr* h, size_t n) {
        OpTimer ot_(c, "vwrite");
        if (at + n > v.n) throw MarlinError("vwrite: range out of bounds");
        if (n) {
            cu(cudaMemcpyAsync(v.p + at, h, n * sizeof(Fr), cudaMemcpyHostToDevice, c->stream), "H2D");
            cu(cudaStreamSynchronize(c->stream), "sync");     // h may be a temporary
        }
    }
    std::vector<Fr> vhost(const Vec& v) {
        OpTimer ot_(c, "vhost");
        std::vector<Fr> h(v.n);
        if (v.n) {
            cu(cudaMemcpyAsync(h.data(), v.p, v.n * sizeof(Fr), cudaMemcpyDeviceToHost, c->stream), "D2H");
            cu(cudaStreamSynchronize(c->stream), "sync");
        }
        return h;
    }
    Vec vclone(const Vec& v) {
        OpTimer ot_(c, "vclone");
        Vec r = alloc(v.n);
        if (v.n) cu(cudaMemcpyAsync(r.p, v.p, v.n * sizeof(Fr), cudaMemcpyDeviceToDevice, c->stream), "D2D");
        return r;
    }
    void vresize(Vec& v, size_t n) {
        OpTimer ot_(c, "vresize");
        if (!v.c) v.c = c;
        if (n <= v.cap) {
            if (n > v.n) cu(cudaMemsetAsync(v.p + v.n, 0, (n - v.n) * sizeof(Fr), c->stream), "memset");
            v.n = n;
            return;
        }
        Vec r = alloc(n);
        if (v.n) cu(cudaMemcpyAsync(r.p, v.p, v.n * sizeof(Fr), cudaMemcpyDeviceToDevice, c->stream), "D2D");
        cu(cudaMemsetAsync(r.p + v.n, 0, (n - v.n) * sizeof(Fr), c->stream), "memset");
        v = std::move(r);
    }
    size_t vlen(const Vec& v) {
        OpTimer ot_(c, "vlen");
        size_t len = 0;
        ck(poly_len_dev(c, v.p, v.n, &len), "poly_len");
        return len;
    }
    Fr vget(const Vec& v, size_t i) {
        OpTimer ot_(c, "vget");
        if (i >= v.n) throw MarlinError("vget: index out of range");
        Fr x;
        cu(cudaMemcpyAsync(&x, v.p + i, sizeof(Fr), cudaMemcpyDeviceToHost, c->stream), "D2H");
        cu(cudaStreamSynchronize(c->stream), "sync");
        return x;
    }
    void vset(Vec& v, size_t i, const Fr& x) {
        OpTimer ot_(c, "vset");
        if (i >= v.n) throw MarlinError("vset: index out of range");
        cu(cudaMemcpyAsync(v.p + i, &x, sizeof(Fr), cudaMemcpyHostToDevice, c->stream), "H2D");
        cu(cudaStreamSynchronize(c->stream), "sync");
    }
    // ---- element-wise ---------------------------------------------------------------------------
    void vmul(Vec& a, const Vec& b) {
        OpTimer ot_(c, "vmul");
        if (a.n != b.n) throw MarlinError("vmul: size mismatch");
        ck(poly_mul_ew(c, a.p, b.p, a.n), "vmul");
    }
    void vadd(Vec& a, const Vec& b) {
        OpTimer ot_(c, "vadd");
        if (a.n < b.n) vresize(a, b.n);
        ck(poly_add_ew(c, a.p, b.p, b.n), "vadd");
    }
    void vsub(Vec& a, const Vec& b) {
        OpTimer ot_(c, "vsub");
        if (a.n < b.n) vresize(a, b.n);
        ck(poly_sub_ew(c, a.p, b.p, b.n), "vsub");
    }
    void vadd_scaled(Vec& a, const Fr& s, const Vec& b) {
        OpTimer ot_(c, "vadd_scaled");
        if (a.n < b.n) vresize(a, b.n);
        ck(poly_add_scaled_ew(c, a.p, s, b.p, b.n), "vadd_scaled");
    }
    void vscale(Vec& a, const Fr& s) {
        OpTimer ot_(c, "vscale"); ck(poly_scale_ew(c, a.p, s, a.n), "vscale"); }
    void vlin(Vec& a, const Fr& c0, const Fr& c1) {
        OpTimer ot_(c, "vlin"); ck(poly_lin_ew(c, a.p, c0, c1, a.n), "vlin"); }
    void vadd_offset(Vec& a, size_t off, const Vec& b, bool negate) {
        OpTimer ot_(c, "vadd_offset");
        if (a.n < off + b.n) vresize(a, off + b.n);
        ck(negate ? poly_sub_ew(c, a.p + off, b.p, b.n) : poly_add_ew(c, a.p + off, b.p, b.n), "vadd_offset");
    }
    // ---- polynomial -------------------------------------------------------------------------------
    Fr veval(const Vec& p, const Fr& x) {
        OpTimer ot_(c, "veval");
        Fr out;
        ck(poly_eval_dev(c, p.p, p.n, x, &out), "veval");
        return out;
    }
    void vdiv_vanishing(const Vec& p, size_t n, Vec* q, Vec* r) {
        OpTimer ot_(c, "vdiv_vanishing");
        *q = alloc(p.n > n ? p.n - n : 0);
        *r = alloc(n);
        ck(poly_div_vanishing_dev(c, q->p, r->p, p.p, p.n, n), "vdiv_vanishing");
    }
    Vec vdiv_linear(const Vec& p, const Fr& z) {
        OpTimer ot_(c, "vdiv_linear");
        Vec q = alloc(p.n > 1 ? p.n - 1 : 0);
        ck(poly_div_linear_dev(c, q.p, p.p, p.n, z), "vdiv_linear");
        return q;
    }
    void vbatch_inverse(Vec& v) {
        OpTimer ot_(c, "vbatch_inverse"); ck(swb_fr_batch_inverse_dev(c, reinterpret_cast<swb_fr*>(v.p), v.n), "vbatch_inverse"); }
    Vec vshift_down(const Vec& p, size_t k) {
        OpTimer ot_(c, "vshift_down");
        if (k >= p.n) return alloc(0);
        Vec r = alloc(p.n - k);
        cu(cudaMemcpyAsync(r.p, p.p + k, (p.n - k) * sizeof(Fr), cudaMemcpyDeviceToDevice, c->stream), "D2D");
        return r;
    }
    Vec vdomain(uint32_t log_n) {
        OpTimer ot_(c, "vdomain");
        Vec r = alloc((size_t)1 << log_n);
        ck(poly_powers_dev(c, r.p, r.n, Domain((size_t)1 << log_n).gen), "vdomain");
        return r;
    }
    void vntt(Vec& v, uint32_t log_n, bool inverse, bool coset) {
        OpTimer ot_(c, "vntt");
        if (v.n != ((size_t)1 << log_n)) throw MarlinError("vntt: size mismatch");
        ck(swb_ntt_fr_dev(c, reinterpret_cast<swb_fr*>(v.p), log_n, inverse, coset), "ntt");
    }
    // ---- prover-specific vectors (marlin_ops.cu) ----------------------------------------------------
    Vec vrand(ChaChaRng& rng, size_t n) {
        OpTimer ot_(c, "vrand");
        Vec v = alloc(n);
        uint64_t used = 0;
        ck(rand_fr_dev(c, v.p, n, rng.key_words(), rng.rounds(), rng.position(), &used), "vrand");
        rng.seek(rng.position() + used);
        return v;
    }
    struct DevCsr {
        uint32_t *start = nullptr, *col = nullptr;
        Fr* coef = nullptr;
        uint8_t* tag = nullptr;
        size_t nrows = 0, nnz = 0;
    };
    template <class T>
    T* upload(const std::vector<T>& h) {
        T* d = nullptr;
        cu(cudaMalloc((void**)&d, (h.size() ? h.size() : 1) * sizeof(T)), "cudaMalloc");
        if (!h.empty()) cu(cudaMemcpyAsync(d, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice, c->stream), "H2D");
        return d;
    }
    void* csr_upload(const std::vector<uint32_t>& start, const std::vector<uint32_t>& col, const std::vector<Fr>& coef,
                     const std::vector<uint8_t>* tag) {
        DevCsr* m = new DevCsr();
        m->nrows = start.size() - 1;
        m->nnz = col.size();
        m->start = upload(start);
        m->col = upload(col);
        m->coef = upload(coef);
        if (tag) m->tag = upload(*tag);
        cu(cudaStreamSynchronize(c->stream), "sync");        // the host vectors may be temporaries
        return m;
    }
    // The same, with the column and coefficient arrays written by `fill(col, coef)` straight into the context's pinned
    // staging buffer: no zero-initialised host vectors (page faults on 40 MB per matrix at 2^20 rows) and the copy runs at
    // the link's rate instead of the pageable path's.
    template <class Fill>
    void* csr_upload_filled(const std::vector<uint32_t>& start, Fill&& fill) {
        const size_t nnz = start.back();
        const size_t coef_off = (nnz * sizeof(uint32_t) + 63) & ~(size_t)63;
        char* st = static_cast<char*>(get_pinned(c, coef_off + nnz * sizeof(Fr) + 64));
        if (!st) ck(SWB_ENOMEM, "index (pinned staging)");
        uint32_t* col = reinterpret_cast<uint32_t*>(st);
        Fr* coef = reinterpret_cast<Fr*>(st + coef_off);
        fill(col, coef);
        DevCsr* m = new DevCsr();
        m->nrows = start.size() - 1;
        m->nnz = nnz;
        m->start = upload(start);
        cu(cudaMalloc((void**)&m->col, (nnz ? nnz : 1) * sizeof(uint32_t)), "cudaMalloc");
        cu(cudaMalloc((void**)&m->coef, (nnz ? nnz : 1) * sizeof(Fr)), "cudaMalloc");
        if (nnz) {
            cu(cudaMemcpyAsync(m->col, col, nnz * sizeof(uint32_t), cudaMemcpyHostToDevice, c->stream), "H2D");
            cu(cudaMemcpyAsync(m->coef, coef, nnz * sizeof(Fr), cudaMemcpyHostToDevice, c->stream), "H2D");
        }
        cu(cudaStreamSynchronize(c->stream), "sync");        // the staging buffer is reused by the next matrix
        return m;
    }
    // Marlin's index arithmetisation on the device (index_ops.cu): joint sparsity pattern of the three uploaded matrices,
    // the six evaluation vectors on K and the column-grouped copy for the prover's t polynomial
    static constexpr bool kDeviceIndex = true;
    struct IndexOut { size_t nnz = 0; Vec row, col, va, vb, vc, rowcol; void* m_t = nullptr; };
    IndexOut index_arith(void* ha, void* hb, void* hc, size_t ncons, size_t nvar, size_t ninst, const Domain& H) {
        OpTimer ot_(c, "index_arith");
        const DevCsr* ms[3] = {static_cast<DevCsr*>(ha), static_cast<DevCsr*>(hb), static_cast<DevCsr*>(hc)};
        IndexCsr in[3];
        for (int w = 0; w < 3; w++) {
            in[w].start = ms[w]->start; in[w].col = ms[w]->col; in[w].coef = ms[w]->coef; in[w].nnz = ms[w]->nnz;
        }
        if (ncons >= ((size_t)1 << 31) || nvar >= ((size_t)1 << 31)) throw MarlinError("index: constraint system too large");
        IndexJoint j;
        ck(index_joint_dev(c, in, (uint32_t)ncons, (uint32_t)nvar, (uint32_t)ninst, (uint32_t)H.n, &j), "index (joint pattern)");
        IndexOut out;
        out.nnz = j.nnz;
        out.row = alloc(j.kn); out.col = alloc(j.kn); out.va = alloc(j.kn); out.vb = alloc(j.kn); out.vc = alloc(j.kn);
        out.rowcol = alloc(j.kn);
        Vec hel = vdomain(H.log_n);
        DevCsr* t = new DevCsr();
        t->nrows = H.n;
        t->nnz = j.total;
        cu(cudaMalloc((void**)&t->start, (H.n + 1) * sizeof(uint32_t)), "cudaMalloc");
        cu(cudaMalloc((void**)&t->col, ((size_t)j.total + 1) * sizeof(uint32_t)), "cudaMalloc");
        cu(cudaMalloc((void**)&t->coef, ((size_t)j.total + 1) * sizeof(Fr)), "cudaMalloc");
        cu(cudaMalloc((void**)&t->tag, (size_t)j.total + 1), "cudaMalloc");
        out.m_t = t;
        ck(index_fill_dev(c, in, (uint32_t)ncons, (uint32_t)ninst, (uint32_t)H.n, j, hel.p, H.size_inv, out.row.p, out.col.p, out.va.p,
                          out.vb.p, out.vc.p, out.rowcol.p, t->start, t->col, t->tag, t->coef), "index (evaluations)");
        return out;
    }
    void csr_free(void* h) {
        DevCsr* m = static_cast<DevCsr*>(h);
        if (!m) return;
        cudaSetDevice(c->device);
        cudaStreamSynchronize(c->stream);
        cudaFree(m->start); cudaFree(m->col); cudaFree(m->coef); cudaFree(m->tag);
        delete m;
    }
    Vec vspmv(const void* h, const Vec& x, size_t nout, const Fr* weights) {
        OpTimer ot_(c, "vspmv");
        const DevCsr& m = *static_cast<const DevCsr*>(h);
        Vec out = alloc(nout);
        ck(csr_spmv_dev(c, out.p, nout, m.nrows, m.start, m.col, m.coef, m.tag, x.p, weights), "vspmv");
        return out;
    }
    Vec vwitness_evals(const Vec& z, size_t ninst, const Vec& xh_on_h, size_t ratio) {
        OpTimer ot_(c, "vwitness_evals");
        Vec out = alloc(xh_on_h.n);
        ck(witness_evals_dev(c, out.p, xh_on_h.n, ratio, z.p, ninst, z.n, xh_on_h.p), "vwitness_evals");
        return out;
    }
    // ---- bases / MSM --------------------------------------------------------------------------------
    void* bases_from_powers(const G1Point& g, const Fr& beta, size_t n) {
        swb_g1_jacobian gj;
        memset(&gj, 0, sizeof gj);
        Fq one = Fq::one();
        if (g.infinity) memcpy(gj.y.l, one.l, 48);
        else {
            memcpy(gj.x.l, g.x.l, 48);
            memcpy(gj.y.l, g.y.l, 48);
            memcpy(gj.z.l, one.l, 48);
        }
        swb_fr b;
        memcpy(b.l, beta.l, 32);
        swb_bases* out = nullptr;
        ck(swb_bases_from_powers(c, &gj, &b, n, &out), "bases_from_powers");
        return out;
    }
    // resident bases from host points (a deserialised committer key)
    void* bases_load(const std::vector<G1Point>& pts) {
        std::vector<swb_g1_affine> tmp(pts.size());
        for (size_t i = 0; i < pts.size(); i++) {
            memset(&tmp[i], 0, sizeof tmp[i]);
            if (pts[i].infinity) tmp[i].infinity = 1;
            else {
                memcpy(tmp[i].x.l, pts[i].x.l, 48);
                memcpy(tmp[i].y.l, pts[i].y.l, 48);
            }
        }
        swb_bases* out = nullptr;
        ck(swb_bases_load(c, tmp.data(), tmp.size(), &out), "bases_load");
        return out;
    }
    // a device-resident CSR matrix back on the host (proving-key serialisation)
    void csr_download(const void* h, std::vector<uint32_t>* start, std::vector<uint32_t>* col, std::vector<Fr>* coef) {
        const DevCsr& m = *static_cast<const DevCsr*>(h);
        start->resize(m.nrows + 1);
        col->resize(m.nnz);
        coef->resize(m.nnz);
        cu(cudaMemcpyAsync(start->data(), m.start, (m.nrows + 1) * sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream), "D2H");
        if (m.nnz) {
            cu(cudaMemcpyAsync(col->data(), m.col, m.nnz * sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream), "D2H");
            cu(cudaMemcpyAsync(coef->data(), m.coef, m.nnz * sizeof(Fr), cudaMemcpyDeviceToHost, c->stream), "D2H");
        }
        cu(cudaStreamSynchronize(c->stream), "sync");
    }
    void export_bases(void* h, size_t offset, size_t n, G1Point* out) {
        std::vector<swb_g1_affine> tmp(n);
        ck(swb_bases_export(c, static_cast<swb_bases*>(h), offset, n, tmp.data()), "bases_export");
        for (size_t i = 0; i < n; i++) {
            out[i].infinity = tmp[i].infinity != 0;
            memcpy(out[i].x.l, tmp[i].x.l, 48);
            memcpy(out[i].y.l, tmp[i].y.l, 48);
        }
    }
    void free_bases(void* h) { swb_bases_free(static_cast<swb_bases*>(h)); }
    // window tables (swb_bases_precompute) with the digit width that suits MSMs of about typical_n
    // scalars (tables_pick_window).  KZG powers lie in the prime-order subgroup (g is cofactor-cleared), which the
    // tables require.
    // Skipped silently when they would not fit in half of the free device memory.
    void bases_tune(void* h, size_t typical_n) {
        swb_bases* b = static_cast<swb_bases*>(h);
        if (!b || typical_n == 0) return;
        const int best = tables_pick_window(typical_n);
        const size_t W = (253 + best - 1) / best;
        size_t free_b = 0, total_b = 0;
        cudaSetDevice(c->device);
        if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess || swb_bases_len(b) * W * 96 > free_b / 2) {
            if (c->trace) fprintf(stderr, "[swb trace] SRS window tables skipped: %zu B needed, %zu B free\n", swb_bases_len(b) * W * 96, free_b);
            return;
        }
        if (swb_bases_precompute(c, b, best) != SWB_OK) {                     // keep going on the plain path
            cudaGetLastError();
            if (c->trace) fprintf(stderr, "[swb trace] SRS window tables not built: %s\n", swb_last_error(c));
        }
    }
    // Independent MSMs (the commitments of a round, the parts of an opening) are submitted first and
    // collected later: two of them are in flight on the library's MSM slots, so the latency-bound
    // bucket tail of one runs under the accumulation of the next.  The scalars must stay alive until the
    // result has been collected.
    // An MSM is first only NOTED (its scalars must stay alive until the result has been collected); the list is
    // launched when a result is asked for: over window tables as ONE batched pipeline (msm_begin_batch: one sort, one
    // accumulation, one bucket reduction for all commitments of a prover round), otherwise one after the other on the
    // library's two MSM slots, whose bucket tails overlap with the next accumulation.
    struct Ticket {
        void* h; size_t offset; const Fr* scalars; size_t n;     // the request
        bool launched, done, sharded, combined, by_bucket;
        int slot;
        G1Point value;
        swb_g1_jacobian share;
    };
    std::vector<Ticket> tickets;                           // ids ticket_base .. ; finished old ones are dropped in blocks
    size_t ticket_base = 0;
    long slot_owner[swb_ctx::MSM_SLOTS] = {-1, -1, -1};    // ticket id occupying each slot
    int next_slot = 1;
    static G1Point from_jacobian(const swb_g1_jacobian& out) {
        G1Point p = G1Point::identity();
        Fq z;
        memcpy(z.l, out.z.l, 48);
        if (!z.is_zero()) {                 // the library returns Z = 1
            p.infinity = false;
            memcpy(p.x.l, out.x.l, 48);
            memcpy(p.y.l, out.y.l, 48);
        }
        return p;
    }
    bool sharding() const { return c->shard_world > 1 && (c->shard_combine || c->comm); }
    // Power-of-two worlds shard by BUCKET (swb::BucketShard: every rank sees the whole polynomial -- it
    // has it anyway -- and fills its interleaved share of the buckets, so accumulation AND bucket reduction shrink
    // and the window width stays that of one GPU); other worlds by contiguous index range.
    bool shards_by_bucket() const { return sharding() && (c->shard_world & (c->shard_world - 1)) == 0; }
    // (only over bases with window tables: on the plain path every rank would still sort all pairs, and the index
    // split measured slightly faster -- 2^20 constraints on two GPUs: 0.248 s against 0.256 s)
    bool bucket_mode(const swb_bases* b) const { return shards_by_bucket() && b && b->tab_w > 0; }
    // the bucket shard ticket t runs under: this rank's share for a by-bucket ticket, else the context's own
    BucketShard bucket_shard(const Ticket& t) const {
        return t.by_bucket ? BucketShard{c->shard_rank, c->shard_world} : BucketShard{c->bucket_rank, c->bucket_world};
    }
    void finish(Ticket& t) {
        t.done = true;
        if (!t.sharded) {
            t.value = from_jacobian(t.share);
            t.combined = true;
        }
    }
    // this rank's part of ticket t as (offset, scalars, n)
    void local_part(const Ticket& t, size_t* off, const Fr** sc, size_t* n) const {
        *off = t.offset; *sc = t.scalars; *n = t.n;
        if (t.sharded && !t.by_bucket) {       // contiguous share of the index range (remainder to the first ranks)
            const size_t base = t.n / (size_t)c->shard_world, rem = t.n % (size_t)c->shard_world, r = (size_t)c->shard_rank;
            const size_t lo = r * base + (r < rem ? r : rem);
            *off = t.offset + lo; *sc = t.scalars + lo; *n = base + (r < rem ? 1 : 0);
        }
    }
    void launch_single(size_t id) {
        Ticket& t = tickets.at(id - ticket_base);
        const int slot = next_slot;
        next_slot = next_slot == 1 ? 2 : 1;
        if (slot_owner[slot] >= 0) collect((size_t)slot_owner[slot]);
        size_t off, n;
        const Fr* sc;
        local_part(t, &off, &sc, &n);
        ck(msm_begin(c, slot, static_cast<swb_bases*>(t.h), off, sc, n, 1, bucket_shard(t)), "msm");
        t.launched = true;
        t.slot = slot;
        slot_owner[slot] = (long)id;
    }
    // launches every noted ticket; runs of tickets over the same table-backed handle go out as batches
    void flush() {
        size_t k = 0;
        while (k < tickets.size()) {
            if (tickets[k].launched) { k++; continue; }
            size_t e = k;
            std::vector<size_t> offs, ns;
            std::vector<const void*> scs;
            while (e < tickets.size() && !tickets[e].launched && tickets[e].h == tickets[k].h &&
                   tickets[e].sharded == tickets[k].sharded && tickets[e].by_bucket == tickets[k].by_bucket && e - k < (size_t)MSM_MAX_BATCH) {
                size_t off, n;
                const Fr* sc;
                local_part(tickets[e], &off, &sc, &n);
                offs.push_back(off); ns.push_back(n); scs.push_back(sc);
                e++;
            }
            swb_bases* b = static_cast<swb_bases*>(tickets[k].h);
            if (e - k >= 2 && msm_can_batch(c, b, e - k, ns.data())) {
                // the slots must be idle: the batch runs on the context's stream with slot 0's scratch
                for (int sl = 1; sl < swb_ctx::MSM_SLOTS; sl++)
                    if (slot_owner[sl] >= 0) collect((size_t)slot_owner[sl]);
                ck(msm_begin_batch(c, 0, b, e - k, offs.data(), scs.data(), ns.data(), 1, bucket_shard(tickets[k])), "msm (batch)");
                std::vector<swb_g1_jacobian> outs(e - k);
                ck(msm_end(c, 0, outs.data()), "msm (batch)");
                for (size_t q = k; q < e; q++) {
                    tickets[q].launched = true;
                    tickets[q].slot = 0;
                    tickets[q].share = outs[q - k];
                    finish(tickets[q]);
                }
            } else {
                for (size_t q = k; q < e; q++) launch_single(ticket_base + q);
            }
            k = e;
        }
    }
    // finishes the local part of a ticket (this rank's share when sharded)
    void collect(size_t id) {
        Ticket& t = tickets.at(id - ticket_base);
        if (t.done) return;
        if (!t.launched) flush();
        if (t.done) return;
        ck(msm_end(c, t.slot, &t.share), "msm");
        slot_owner[t.slot] = -1;
        finish(t);
    }
    // shares -> sums over all ranks.  With the library's communicator every share that is outstanding (the
    // commitments of a round are all submitted before the first result is asked for) goes into ONE all-gather;
    // a caller-supplied callback is invoked per MSM.
    void combine_pending() {
        std::vector<size_t> ids;
        for (size_t k = 0; k < tickets.size(); k++)
            if (tickets[k].sharded && !tickets[k].combined) ids.push_back(ticket_base + k);
        if (ids.empty()) return;
        for (size_t id : ids) collect(id);
        if (c->shard_combine) {
            for (size_t id : ids) {
                Ticket& t = tickets.at(id - ticket_base);
                swb_g1_jacobian sum;
                if (c->shard_combine(c->shard_user, &t.share, &sum) != 0) throw MarlinError("msm: combining the ranks' partial results failed");
                t.value = from_jacobian(sum);
                t.combined = true;
            }
            return;
        }
        std::vector<swb_g1_jacobian> mine(ids.size()), sums(ids.size());
        for (size_t k = 0; k < ids.size(); k++) mine[k] = tickets.at(ids[k] - ticket_base).share;
        ck(comm_sum_g1(c, mine.data(), mine.size(), sums.data()), "msm (all-gather of the partial results)");
        for (size_t k = 0; k < ids.size(); k++) {
            Ticket& t = tickets.at(ids[k] - ticket_base);
            t.value = from_jacobian(sums[k]);
            t.combined = true;
        }
    }
    // (sizes the SRS window tables: in a power-of-two world they will be used by bucket, i.e. on whole polynomials)
    size_t msm_local_count(size_t n) {
        if (!sharding() || shards_by_bucket()) return n;
        const size_t base = n / (size_t)c->shard_world, rem = n % (size_t)c->shard_world;
        return base + ((size_t)c->shard_rank < rem ? 1 : 0);
    }
    size_t msm_submit(void* h, size_t offset, const Vec& scalars, size_t n) {
        OpTimer ot_(c, "msm_submit");
        if (tickets.size() >= 128) {                       // batches are a handful of MSMs: these are long finished
            for (size_t i = 0; i < 64; i++) collect(ticket_base + i);
            combine_pending();
            tickets.erase(tickets.begin(), tickets.begin() + 64);
            ticket_base += 64;
        }
        Ticket t{};
        t.h = h; t.offset = offset; t.scalars = scalars.p; t.n = n;
        t.sharded = sharding();
        t.by_bucket = bucket_mode(static_cast<swb_bases*>(h));
        t.slot = -1;
        t.value = G1Point::identity();
        tickets.push_back(t);
        return ticket_base + tickets.size() - 1;
    }
    G1Point msm_result(size_t id) {
        OpTimer ot_(c, "msm_result");
        collect(id);
        if (!tickets.at(id - ticket_base).combined) combine_pending();
        return tickets.at(id - ticket_base).value;
    }
    void msm_drain() {
        for (size_t i = 0; i < tickets.size(); i++) collect(ticket_base + i);
        combine_pending();
    }
    ~GpuEngine() {
        try { msm_drain(); } catch (...) {}
    }
};
using Api = MarlinApi<GpuEngine>;

}  // namespace

struct swb_rng { RngHandle h; };
struct swb_r1cs { R1csHandle* h; };
// A proving key points into the SRS it was indexed from (committer key, engine), so the SRS is reference
// counted: swb_srs_free only drops the caller's reference and the last proving key releases the rest.
struct swb_srs { GpuEngine eng; SrsHandle<GpuEngine>* h; swb_ctx* ctx; int refs; };
struct swb_pk { PkHandle<GpuEngine>* h; swb_srs* srs; };
static void srs_release(swb_srs* s) {
    if (!s || --s->refs > 0) return;
    delete s->h;
    delete s;
}
struct swb_vk { VkHandle* h; };
struct swb_proof { Proof p; };

extern "C" {

swb_rng* swb_rng_test_rng(void) {
    auto* r = new swb_rng();
    r->h.rng = test_rng();
    return r;
}
swb_rng* swb_rng_from_seed(const uint8_t seed[32]) {
    if (!seed) return nullptr;
    auto* r = new swb_rng();
    r->h.rng = ChaChaRng(seed, 12);
    return r;
}
swb_rng* swb_rng_from_entropy(void) {
    uint8_t seed[32];
    if (!os_entropy(seed)) return nullptr;
    return swb_rng_from_seed(seed);
}
uint64_t swb_rng_next_u64(swb_rng* r) { return r->h.rng.next_u64(); }
void swb_rng_free(swb_rng* r) { delete r; }

swb_r1cs* swb_r1cs_new(size_t num_instance, size_t num_witness) { return new swb_r1cs{r1cs_new(num_instance, num_witness)}; }
swb_r1cs* swb_r1cs_builtin(int kind, size_t size, uint64_t v0, uint64_t v1) {
    R1csHandle* h = r1cs_builtin(kind, size, v0, v1);
    return h ? new swb_r1cs{h} : nullptr;
}
int swb_r1cs_add_constraint(swb_r1cs* cs, const swb_fr* a_coef, const uint32_t* a_col, size_t na, const swb_fr* b_coef,
                            const uint32_t* b_col, size_t nb, const swb_fr* c_coef, const uint32_t* c_col, size_t nc) {
    if (!cs) return SWB_EARG;
    return r1cs_add_constraint(cs->h, (const uint64_t*)a_coef, a_col, na, (const uint64_t*)b_coef, b_col, nb, (const uint64_t*)c_coef,
                               c_col, nc) ? SWB_EARG : SWB_OK;
}
int swb_r1cs_set_assignment(swb_r1cs* cs, const swb_fr* instance, size_t ni, const swb_fr* witness, size_t nw) {
    if (!cs) return SWB_EARG;
    return r1cs_set_assignment(cs->h, (const uint64_t*)instance, ni, (const uint64_t*)witness, nw) ? SWB_EARG : SWB_OK;
}
int swb_r1cs_is_satisfied(const swb_r1cs* cs) { return cs && cs->h->cs.is_satisfied() ? 1 : 0; }
void swb_r1cs_free(swb_r1cs* cs) {
    if (!cs) return;
    delete cs->h;
    delete cs;
}

int swb_marlin_profile_enable(int enable) {
    HostProfile& hp = host_profile();
    hp.on = enable != 0 || hp.print;
    if (!hp.on) hp.acc.clear();
    return SWB_OK;
}
size_t swb_marlin_last_phases(char* buf, size_t cap) {
    const std::string& s = host_profile().last;
    if (buf && cap) {
        const size_t k = s.size() < cap - 1 ? s.size() : cap - 1;
        memcpy(buf, s.data(), k);
        buf[k] = 0;
    }
    return s.size() + 1;
}

int swb_marlin_universal_setup(swb_ctx* c, size_t nc, size_t nv, size_t nnz, swb_rng* rng, swb_srs** out) {
    if (!c || !rng || !out) return SWB_EARG;
    auto* s = new swb_srs{GpuEngine(c), nullptr, c, 1};
    std::string err;
    int rc = Api::setup(s->eng, nc, nv, nnz, &rng->h, &s->h, &err);
    if (rc) {
        delete s;
        return swb::set_err(c, SWB_EINTERNAL, "universal_setup: %s", err.c_str());
    }
    *out = s;
    return SWB_OK;
}
size_t swb_srs_max_degree(const swb_srs* s) { return s ? s->h->srs->max_degree : 0; }
int swb_srs_set_tune_after(swb_srs* s, long n_msms) {
    if (!s || n_msms < 0) return SWB_EARG;
    s->h->srs->tune_after = n_msms;
    return SWB_OK;
}
int swb_srs_table_info(const swb_srs* s, int* window_bits, int* levels) {
    if (!s) return SWB_EARG;
    return swb_bases_table_info(static_cast<const swb_bases*>(s->h->srs->powers_of_g), window_bits, levels);
}
void swb_srs_free(swb_srs* s) { srs_release(s); }
int swb_marlin_index(swb_ctx* c, const swb_srs* srs, const swb_r1cs* cs, swb_pk** pk, swb_vk** vk) {
    if (!c || !srs || !cs || !pk || !vk) return SWB_EARG;
    if (srs->ctx != c) return swb::set_err(c, SWB_EARG, "%s", "index: the SRS was built on another context");
    std::string err;
    auto* p = new swb_pk{nullptr, nullptr};
    auto* v = new swb_vk{nullptr};
    GpuEngine eng(c);
    int rc = Api::index(eng, srs->h, cs->h, &p->h, &v->h, &err);
    if (rc) {
        delete p;
        delete v;
        return swb::set_err(c, SWB_EINTERNAL, "index: %s", err.c_str());
    }
    p->srs = const_cast<swb_srs*>(srs);
    p->srs->refs++;
    *pk = p;
    *vk = v;
    return SWB_OK;
}
void swb_pk_free(swb_pk* p) {
    if (!p) return;
    delete p->h;                 // releases the device-resident matrices through the SRS's engine ...
    srs_release(p->srs);         // ... which therefore goes last
    delete p;
}
void swb_vk_free(swb_vk* v) {
    if (!v) return;
    delete v->h;
    delete v;
}
int swb_marlin_prove(swb_ctx* c, const swb_pk* pk, const swb_r1cs* cs, swb_rng* rng, uint8_t** proof, size_t* len) {
    if (!c || !pk || !cs || !rng || !proof || !len) return SWB_EARG;
    if (pk->srs && pk->srs->ctx != c) return swb::set_err(c, SWB_EARG, "%s", "prove: the proving key belongs to another context");
    std::string err;
    GpuEngine eng(c);
    int rc = Api::prove(eng, pk->h, cs->h, &rng->h, proof, len, &err);
    if (rc) return swb::set_err(c, SWB_EINTERNAL, "prove: %s", err.c_str());
    return SWB_OK;
}
int swb_marlin_verify(swb_ctx* c, const swb_vk* vk, const swb_fr* public_inputs, size_t n, const uint8_t* proof, size_t len,
                      swb_rng* rng, int* ok) {
    if (!vk || !ok || (!public_inputs && n) || !proof) return SWB_EARG;
    std::string err;
    int rc = Api::verify(vk->h, (const uint64_t*)public_inputs, n, proof, len, rng ? &rng->h : nullptr, ok, &err);
    if (rc) return swb::set_err(c, SWB_EINTERNAL, "verify: %s", err.c_str());
    return SWB_OK;
}
void swb_bytes_free(uint8_t* p) { free(p); }

swb_r1cs* swb_r1cs_read(const uint8_t* bytes, size_t len) {
    R1csHandle* h = bytes ? r1cs_from_bytes(bytes, len) : nullptr;
    return h ? new swb_r1cs{h} : nullptr;
}
int swb_r1cs_write(const swb_r1cs* cs, uint8_t** bytes, size_t* len) {
    if (!cs || !bytes || !len) return SWB_EARG;
    *bytes = r1cs_to_bytes(cs->h, len);
    return SWB_OK;
}
int swb_vk_serialize(const swb_vk* vk, uint8_t** bytes, size_t* len) {
    if (!vk || !bytes || !len) return SWB_EARG;
    *bytes = vk_to_bytes(vk->h, len);
    return SWB_OK;
}
swb_vk* swb_vk_deserialize(const uint8_t* bytes, size_t len) {
    VkHandle* h = bytes ? vk_from_bytes(bytes, len) : nullptr;
    return h ? new swb_vk{h} : nullptr;
}

// ---- proofs as objects (deserialize_proof / serialize_proof, reference src/marlin/serialization.rs:5-17) ----------
swb_proof* swb_proof_deserialize(const uint8_t* bytes, size_t len) {
    if (!bytes) return nullptr;
    swb_proof* p = nullptr;
    try {
        p = new swb_proof();
        if (!Proof::deserialize(bytes, len, &p->p)) { delete p; return nullptr; }
        return p;
    } catch (...) {
        delete p;
        return nullptr;
    }
}
int swb_proof_serialize(const swb_proof* proof, uint8_t** bytes, size_t* len) {
    if (!proof || !bytes || !len) return SWB_EARG;
    *bytes = bytes_out(proof->p.serialize(), len);
    return SWB_OK;
}
void swb_proof_free(swb_proof* p) { delete p; }
int swb_marlin_verify_proof(swb_ctx* c, const swb_vk* vk, const swb_fr* public_inputs, size_t n, const swb_proof* proof, swb_rng* rng,
                            int* ok) {
    if (!vk || !ok || (!public_inputs && n) || !proof) return SWB_EARG;
    size_t len = 0;
    uint8_t* b = bytes_out(proof->p.serialize(), &len);
    const int rc = swb_marlin_verify(c, vk, public_inputs, n, b, len, rng, ok);
    free(b);
    return rc;
}

// ---- proving keys (serialize_proving_key / deserialize_proving_key, serialization.rs:33-45) -------------------------
// "SWBPK001" | u64 max_degree | g, gamma_g (97 B each) | h, beta_h (96 B compressed) | 3 powers of gamma_g (97 B) |
// u64 n | n powers of g as raw Montgomery (x, y) pairs, 96 B each (the committer key; raw because decompressing
// millions of points costs a square root each) | u64 len, verifying-key bytes | u64 len, SWBR1CS1 bytes of the padded,
// squared constraint matrices (no assignment).  Like upstream, the key carries its committer key and needs no SRS to be
// loaded again; unlike upstream the layout is this library's own (arkworks' is unpinned here, DESIGN.md section 2).
// Loading re-derives the index on the device from the matrices and refuses the key unless the verifying key it obtains
// is byte-identical to the stored one.
int swb_pk_serialize(swb_ctx* c, const swb_pk* pk, const swb_vk* vk, uint8_t** bytes, size_t* len) {
    if (!c || !pk || !vk || !bytes || !len || !pk->srs) return SWB_EARG;
    if (pk->srs->ctx != c) return swb::set_err(c, SWB_EARG, "%s", "pk_serialize: the proving key belongs to another context");
    try {
        GpuEngine eng(c);
        const UniversalSrs<GpuEngine>& srs = *pk->srs->h->srs;
        const ProvingKey<GpuEngine>& k = pk->h->pk;
        std::vector<uint8_t> out;
        const char magic[8] = {'S', 'W', 'B', 'P', 'K', '0', '0', '1'};
        out.insert(out.end(), magic, magic + 8);
        put_u64(out, srs.max_degree);
        put_g1_uncompressed(out, srs.g);
        put_g1_uncompressed(out, srs.gamma_g);
        put_g2_compressed(out, srs.h);
        put_g2_compressed(out, srs.beta_h);
        if (srs.powers_of_gamma_g.size() != 3) throw MarlinError("pk_serialize: unexpected committer key");
        for (auto& gp : srs.powers_of_gamma_g) put_g1_uncompressed(out, gp);
        const size_t np = srs.max_degree + 1;
        put_u64(out, np);
        {
            const size_t at = out.size();
            out.resize(at + np * 96);
            const size_t chunk = (size_t)1 << 18;
            std::vector<G1Point> tmp(chunk);
            for (size_t i = 0; i < np; i += chunk) {
                const size_t cnt = np - i < chunk ? np - i : chunk;
                eng.export_bases(srs.powers_of_g, i, cnt, tmp.data());
                for (size_t j = 0; j < cnt; j++) {
                    if (tmp[j].infinity) throw MarlinError("pk_serialize: identity among the SRS powers");
                    memcpy(&out[at + (i + j) * 96], tmp[j].x.l, 48);
                    memcpy(&out[at + (i + j) * 96 + 48], tmp[j].y.l, 48);
                }
            }
        }
        const std::vector<uint8_t> vkb = vk->h->vk.serialize();
        put_u64(out, vkb.size());
        out.insert(out.end(), vkb.begin(), vkb.end());
        // the padded, squared matrices as the key holds them on the device
        R1cs cs;
        cs.num_instance = k.info.num_instance;
        cs.num_witness = k.info.num_variables - k.info.num_instance;
        std::vector<SparseRow>* rows[3] = {&cs.a, &cs.b, &cs.c};
        void* ms[3] = {k.m_a, k.m_b, k.m_c};
        for (int w = 0; w < 3; w++) {
            std::vector<uint32_t> start, col;
            std::vector<Fr> coef;
            eng.csr_download(ms[w], &start, &col, &coef);
            rows[w]->resize(k.info.num_constraints);
            for (size_t r = 0; r + 1 < start.size() && r < rows[w]->size(); r++)
                for (uint32_t e = start[r]; e < start[r + 1]; e++) (*rows[w])[r].e.push_back({coef[e], col[e]});
        }
        std::vector<uint8_t> csb;
        r1cs_write(cs, &csb);
        put_u64(out, csb.size());
        out.insert(out.end(), csb.begin(), csb.end());
        *bytes = bytes_out(out, len);
        return SWB_OK;
    } catch (const std::exception& e) {
        return swb::set_err(c, SWB_EINTERNAL, "pk_serialize: %s", e.what());
    }
}

int swb_pk_deserialize(swb_ctx* c, const uint8_t* bytes, size_t len, swb_pk** pk_out, swb_vk** vk_out) {
    if (!c || !bytes || !pk_out) return SWB_EARG;
    swb_srs* s = nullptr;
    swb_pk* p = nullptr;
    swb_vk* v = nullptr;
    try {
        const uint8_t *q = bytes, *end = bytes + len;
        if (len < 8 || memcmp(q, "SWBPK001", 8) != 0) throw MarlinError("bad magic");
        q += 8;
        uint64_t max_degree, np, n;
        if (!get_u64(q, end, &max_degree) || max_degree >= ((uint64_t)1 << 31)) throw MarlinError("bad max_degree");
        auto get_g1_unc = [&](G1Point* out) {
            if (end - q < 97) throw MarlinError("truncated");
            Fq x, y;
            if (!fq_from_canonical_bytes(q, &x) || !fq_from_canonical_bytes(q + 48, &y) || q[96] > 1) throw MarlinError("bad point");
            out->infinity = q[96] != 0;
            out->x = out->infinity ? Fq::zero() : x;
            out->y = out->infinity ? Fq::zero() : y;
            if (!out->infinity && (!(y.sqr() == x.sqr() * x + Fq::one()) || !g1_in_subgroup(*out))) throw MarlinError("point not in G1");
            q += 97;
        };
        s = new swb_srs{GpuEngine(c), new SrsHandle<GpuEngine>(), c, 1};
        s->h->srs.reset(new UniversalSrs<GpuEngine>());
        UniversalSrs<GpuEngine>& srs = *s->h->srs;
        srs.eng = &s->eng;
        srs.max_degree = (size_t)max_degree;
        get_g1_unc(&srs.g);
        get_g1_unc(&srs.gamma_g);
        if (!get_g2_compressed(q, end, &srs.h) || !get_g2_compressed(q, end, &srs.beta_h)) throw MarlinError("bad G2 point");
        srs.powers_of_gamma_g.resize(3);
        for (auto& gp : srs.powers_of_gamma_g) get_g1_unc(&gp);
        if (!get_u64(q, end, &np) || np != max_degree + 1 || (uint64_t)(end - q) / 96 < np) throw MarlinError("bad committer key");
        {
            std::vector<G1Point> pts((size_t)np);
            size_t off_curve = 0;
#pragma omp parallel for schedule(static) reduction(+ : off_curve)
            for (size_t i = 0; i < (size_t)np; i++) {
                memcpy(pts[i].x.l, q + i * 96, 48);
                memcpy(pts[i].y.l, q + i * 96 + 48, 48);
                pts[i].infinity = false;
                // raw Montgomery limbs: reduced and on the curve (the subgroup is not re-checked point by point; the
                // powers an index commits with are bound by the verifying-key comparison below)
                bool ok = true;
                for (int k = 11; k >= 0; k--) {
                    if (pts[i].x.l[k] != FqParams::mod(k)) { ok = pts[i].x.l[k] < FqParams::mod(k); break; }
                    if (k == 0) ok = false;
                }
                for (int k = 11; ok && k >= 0; k--) {
                    if (pts[i].y.l[k] != FqParams::mod(k)) { ok = pts[i].y.l[k] < FqParams::mod(k); break; }
                    if (k == 0) ok = false;
                }
                if (!ok || !(pts[i].y.sqr() == pts[i].x.sqr() * pts[i].x + Fq::one())) off_curve++;
            }
            if (off_curve) throw MarlinError("committer key holds points that are not on the curve");
            q += (size_t)np * 96;
            srs.powers_of_g = s->eng.bases_load(pts);
        }
        if (!get_u64(q, end, &n) || (uint64_t)(end - q) < n) throw MarlinError("truncated verifying key");
        const std::vector<uint8_t> vkb(q, q + n);
        q += n;
        if (!get_u64(q, end, &n) || (uint64_t)(end - q) != n) throw MarlinError("truncated constraint matrices");
        std::unique_ptr<R1csHandle> cs(r1cs_from_bytes(q, (size_t)n));
        if (!cs) throw MarlinError("malformed constraint matrices");
        // re-derive the index on the device; the stored verifying key is the integrity check (it binds the matrices, the
        // committer key and the index commitments together)
        p = new swb_pk{nullptr, nullptr};
        v = new swb_vk{nullptr};
        GpuEngine eng(c);
        std::string err;
        if (Api::index(eng, s->h, cs.get(), &p->h, &v->h, &err)) throw MarlinError("index: " + err);
        if (v->h->vk.serialize() != vkb) throw MarlinError("the key does not reproduce its verifying key");
        p->srs = s;                 // the key owns the only reference to its committer key
        *pk_out = p;
        if (vk_out) *vk_out = v;
        else swb_vk_free(v);
        return SWB_OK;
    } catch (const std::exception& e) {
        if (p) { delete p->h; delete p; }
        if (v) swb_vk_free(v);
        if (s) srs_release(s);
        return swb::set_err(c, SWB_EINTERNAL, "pk_deserialize: %s", e.what());
    }
}

}  // extern "C"
