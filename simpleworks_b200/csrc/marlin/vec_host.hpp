// Host implementation of the Engine vector interface used by the protocol templates
// (marlin.hpp): Vec = std::vector<Fr> in RAM, every operation (the index arithmetisation included) a
// parallel loop.  The CPU arm (oracle build) derives its engine from this; the CUDA engine
// (marlin_abi.cu) implements the same interface on device memory so that polynomials stay in HBM
// between NTTs and MSMs.
#pragma once
#include <algorithm>
#include <memory>

#include "poly.hpp"
#include "rng.hpp"
#include "curve_host.hpp"

namespace swb {
namespace marlin {

struct HostVecOps {
    using Vec = std::vector<Fr>;
    Vec vzeros(size_t n) { return Vec(n, Fr::zero()); }
    Vec vfrom(const std::vector<Fr>& h) { return h; }
    void vwrite(Vec& v, size_t at, const Fr* p, size_t n) { std::copy(p, p + n, v.begin() + at); }   // v[at .. at+n) = p
    Vec vclone(const Vec& v) { return v; }
    void vresize(Vec& v, size_t n) { v.resize(n, Fr::zero()); }
    size_t vlen(const Vec& v) {
        size_t n = v.size();
        while (n > 0 && v[n - 1].is_zero()) n--;
        return n;
    }
    Fr vget(const Vec& v, size_t i) { return v[i]; }
    void vset(Vec& v, size_t i, const Fr& x) { v[i] = x; }
    void vmul(Vec& a, const Vec& b) {
#pragma omp parallel for schedule(static)
        for (size_t i = 0; i < a.size(); i++) a[i] = a[i] * b[i];
    }
    void vadd(Vec& a, const Vec& b) { poly_add(a, b); }
    void vsub(Vec& a, const Vec& b) { poly_sub(a, b); }
    void vadd_scaled(Vec& a, const Fr& c, const Vec& b) { poly_add_scaled(a, c, b); }
    void vscale(Vec& a, const Fr& c) { poly_scale(a, c); }
    void vlin(Vec& a, const Fr& c0, const Fr& c1) {
#pragma omp parallel for schedule(static)
        for (size_t i = 0; i < a.size(); i++) a[i] = c0 + c1 * a[i];
    }
    // a[off + i] += sign * b[i]
    void vadd_offset(Vec& a, size_t off, const Vec& b, bool negate) {
        if (a.size() < off + b.size()) a.resize(off + b.size(), Fr::zero());
#pragma omp parallel for schedule(static)
        for (size_t i = 0; i < b.size(); i++) a[off + i] = negate ? a[off + i] - b[i] : a[off + i] + b[i];
    }
    Fr veval(const Vec& p, const Fr& x) { return poly_eval(p, x); }
    void vdiv_vanishing(const Vec& p, size_t n, Vec* q, Vec* r) { poly_divide_by_vanishing(p, n, q, r); }
    Vec vdiv_linear(const Vec& p, const Fr& z) { return poly_divide_by_linear(p, z); }
    void vbatch_inverse(Vec& v) { batch_inverse(v); }
    Vec vshift_down(const Vec& p, size_t k) { return k < p.size() ? Vec(p.begin() + k, p.end()) : Vec(); }
    Vec vdomain(uint32_t log_n) { return Domain((size_t)1 << log_n).elements(); }
    // submit / collect interface of the MSM (asynchronous on the CUDA engine): here the derived engine's
    // msm() runs at submission
    std::vector<G1Point> msm_results;     // results of ids msm_base .. ; old ones are dropped in blocks
    size_t msm_base = 0;
    template <class Derived>
    size_t msm_submit_sync(Derived& self, void* h, size_t offset, const Vec& scalars, size_t n) {
        if (msm_results.size() >= 128) {
            msm_results.erase(msm_results.begin(), msm_results.begin() + 64);
            msm_base += 64;
        }
        msm_results.push_back(n ? self.msm(h, offset, scalars, n) : G1Point::identity());
        return msm_base + msm_results.size() - 1;
    }
    G1Point msm_result(size_t id) { return msm_results.at(id - msm_base); }
    size_t msm_local_count(size_t n) { return n; }
    void msm_drain() {}
    // n consecutive Fr::rand draws (DensePolynomial::rand)
    Vec vrand(ChaChaRng& rng, size_t n) {
        Vec v(n);
        rand_fr_bulk(rng, v.data(), n);
        return v;
    }
    // sparse matrices in CSR form (optionally a 0/1/2 tag per entry selecting one of three weights)
    struct HostCsr {
        std::vector<uint32_t> start, col;
        std::vector<Fr> coef;
        std::vector<uint8_t> tag;
    };
    // start [nrows + 1]; the column and coefficient arrays are written by `fill(col, coef)`
    template <class Fill>
    void* csr_upload_filled(const std::vector<uint32_t>& start, Fill&& fill) {
        std::unique_ptr<HostCsr> m(new HostCsr());
        m->start = start;
        m->col.resize(start.back());
        m->coef.resize(start.back());
        fill(m->col.data(), m->coef.data());
        return m.release();
    }
    // Marlin's index arithmetisation (the contract of the CUDA engine's, index_ops.cu) over A, B, C as staged by
    // csr_upload_filled: ncons rows each, columns already shifted by the instance padding.  Returns the joint sparsity
    // pattern's size nnz, the six evaluation vectors on K and the matrices regrouped by the H position of their column
    // (tagged by matrix), for the prover's t.
    struct IndexOut { size_t nnz = 0; Vec row, col, va, vb, vc, rowcol; void* m_t = nullptr; };
    IndexOut index_arith(void* ha, void* hb, void* hc, size_t ncons, size_t nvar, size_t ninst, const Domain& H) {
        const HostCsr* ms[3] = {static_cast<HostCsr*>(ha), static_cast<HostCsr*>(hb), static_cast<HostCsr*>(hc)};
        const Domain X(ninst);
        std::unique_ptr<ScopedPhase> ph(new ScopedPhase("i1_merge_rows"));
        // joint sparsity pattern, row by row, columns in increasing order; rows are independent, so
        // they are merged in parallel: pass 1 counts the distinct columns of each row, pass 2 fills
        struct Ent { uint32_t col; uint8_t which; Fr coef; };
        auto merged_row = [&](size_t r, std::vector<Ent>& tmp) {
            tmp.clear();
            for (uint8_t w = 0; w < 3; w++)
                for (uint32_t e = ms[w]->start[r]; e < ms[w]->start[r + 1]; e++) tmp.push_back(Ent{ms[w]->col[e], w, ms[w]->coef[e]});
            std::stable_sort(tmp.begin(), tmp.end(), [](const Ent& x, const Ent& y) { return x.col < y.col; });
        };
        std::vector<size_t> row_off(ncons + 1, 0);
#pragma omp parallel
        {
            std::vector<Ent> tmp;
#pragma omp for schedule(static)
            for (size_t r = 0; r < ncons; r++) {
                merged_row(r, tmp);
                size_t distinct = 0;
                for (size_t k = 0; k < tmp.size(); k++) distinct += (k == 0 || tmp[k].col != tmp[k - 1].col);
                row_off[r + 1] = distinct;
            }
        }
        for (size_t r = 0; r < ncons; r++) row_off[r + 1] += row_off[r];
        const size_t nnz = row_off[ncons];
        std::vector<uint32_t> er(nnz), ec(nnz);
        std::vector<Fr> sa(nnz, Fr::zero()), sb(nnz, Fr::zero()), sc(nnz, Fr::zero());
#pragma omp parallel
        {
            std::vector<Ent> tmp;
#pragma omp for schedule(static)
            for (size_t r = 0; r < ncons; r++) {
                merged_row(r, tmp);
                size_t at = row_off[r];
                for (size_t k = 0; k < tmp.size(); k++) {
                    if (k && tmp[k].col != tmp[k - 1].col) at++;
                    er[at] = (uint32_t)r;
                    ec[at] = tmp[k].col;
                    Fr& dst = tmp[k].which == 0 ? sa[at] : tmp[k].which == 1 ? sb[at] : sc[at];
                    dst = dst + tmp[k].coef;
                }
            }
        }
        ph.reset();
        // For entry k = (r, c): row_k = H[pos(c)] (the variable side, summed against z), col_k = H[r]
        // (the constraint side, paired with r(alpha, .)).  val_M(k) = M[r][c] / u_H(row_k, row_k) with
        // u_H(x, x) = |H| x^(|H|-1) = |H| / x on H, so that
        //    sum_j z(j) t(j) = sum_r r(alpha, H[r]) (M z)(r)   for   t(X) = sum_k val(k) u_H(X,row_k) u_H(alpha,col_k).
        // Entries past nnz: row = col = H[0], val = 0.
        const size_t kn = Domain(nnz).n;
        const std::vector<Fr> h_el = H.elements();
        IndexOut out;
        out.nnz = nnz;
        out.row = Vec(kn); out.col = Vec(kn); out.va = Vec(kn); out.vb = Vec(kn); out.vc = Vec(kn); out.rowcol = Vec(kn);
#pragma omp parallel for schedule(static)
        for (size_t k = 0; k < kn; k++) {
            if (k >= nnz) {
                out.row[k] = h_el[0]; out.col[k] = h_el[0];
            } else {
                out.row[k] = h_el[H.reindex_by_subdomain(X, ec[k])];
                out.col[k] = h_el[er[k]];
                const Fr scale = out.row[k] * H.size_inv;
                out.va[k] = sa[k] * scale; out.vb[k] = sb[k] * scale; out.vc[k] = sc[k] * scale;
            }
            out.rowcol[k] = out.row[k] * out.col[k];
        }
        ph.reset(new ScopedPhase("i3_transpose"));
        // counting sort of all matrix entries by the H position of their column; the order inside one
        // position is irrelevant (the entries are summed in exact field arithmetic), so both passes run
        // in parallel with atomic cursors
        std::vector<uint32_t> pos_of(nvar), cnt(H.n + 1, 0);
#pragma omp parallel for schedule(static)
        for (size_t v = 0; v < nvar; v++) pos_of[v] = (uint32_t)H.reindex_by_subdomain(X, v);
        for (int w = 0; w < 3; w++) {
            const HostCsr& m = *ms[w];
#pragma omp parallel for schedule(static)
            for (size_t e = 0; e < m.col.size(); e++) {
                uint32_t& slot = cnt[pos_of[m.col[e]] + 1];
#pragma omp atomic
                slot++;
            }
        }
        for (size_t i = 0; i < H.n; i++) cnt[i + 1] += cnt[i];
        std::unique_ptr<HostCsr> t(new HostCsr());
        const size_t tot = cnt[H.n];
        t->col.resize(tot); t->tag.resize(tot); t->coef.resize(tot);
        std::vector<uint32_t> cur(cnt.begin(), cnt.end() - 1);
        for (int w = 0; w < 3; w++) {
            const HostCsr& m = *ms[w];
#pragma omp parallel for schedule(static)
            for (size_t r = 0; r < ncons; r++)
                for (uint32_t e = m.start[r]; e < m.start[r + 1]; e++) {
                    uint32_t at;
                    uint32_t& slot = cur[pos_of[m.col[e]]];
#pragma omp atomic capture
                    at = slot++;
                    t->col[at] = (uint32_t)r; t->tag[at] = (uint8_t)w; t->coef[at] = m.coef[e];
                }
        }
        t->start = std::move(cnt);
        out.m_t = t.release();
        return out;
    }
    void csr_free(void* h) { delete static_cast<HostCsr*>(h); }
    Vec vspmv(const void* h, const Vec& x, size_t nout, const Fr* weights) {
        const HostCsr& m = *static_cast<const HostCsr*>(h);
        const size_t nrows = m.start.size() - 1;
        Vec out(nout, Fr::zero());
#pragma omp parallel for schedule(static)
        for (size_t r = 0; r < nrows; r++) {
            Fr acc = Fr::zero();
            for (uint32_t k = m.start[r]; k < m.start[r + 1]; k++) {
                Fr term = m.coef[k] * x[m.col[k]];
                if (!m.tag.empty()) term = term * weights[m.tag[k]];
                acc = acc + term;
            }
            out[r] = acc;
        }
        return out;
    }
    // w on H before interpolation: 0 on the X-subdomain, witness - x^ elsewhere (z = instance | witness)
    Vec vwitness_evals(const Vec& z, size_t ninst, const Vec& xh_on_h, size_t ratio) {
        const size_t nh = xh_on_h.size();
        Vec out(nh, Fr::zero());
#pragma omp parallel for schedule(static)
        for (size_t k = 0; k < nh; k++) {
            if (k % ratio == 0) continue;
            const size_t wi = ninst + (k - k / ratio - 1);
            out[k] = (wi < z.size() ? z[wi] : Fr::zero()) - xh_on_h[k];
        }
        return out;
    }
};

}  // namespace marlin
}  // namespace swb
