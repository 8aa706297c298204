// Marlin over BLS12-377 with the MarlinKZG10 polynomial commitment: universal setup, index, prove,
// verify -- the protocol that simpleworks::marlin wraps (reference src/marlin/mod.rs:45-94:
// MarlinInst::{universal_setup, index_from_constraint_system, prove_from_constraint_system, verify}).
// The protocol code itself lives in the un-vendored crates ark-marlin (Entropy1729 fork, Cargo.toml:
// 29-30) and ark-poly-commit ^0.3 (Cargo.toml:22); this is a restatement following SURVEY.md
// Appendix A.6-A.10, whose derivation of the AHP identities is repeated next to the code.
// PARITY UNPINNED against real arkworks (no Rust toolchain, no golden proofs in the reference);
// what is checked: completeness (verify(prove(x)) for the reference's toy circuits and synthetic
// ones), soundness smoke tests (tampered proofs / inputs rejected), and that the GPU engine and the
// CPU engine produce byte-identical proofs.
//
// Template parameter Engine supplies the operators and owns the polynomial storage: Engine::Vec is
// a vector of Fr living where the engine computes (HBM for the CUDA engine of libswb200, RAM for
// the CPU arm), so round polynomials stay resident between NTTs, element-wise passes and MSMs.  An SRS
// holds the one engine that serves it (UniversalSrs::eng); index, prove and the proving key use that one.
// What the templates call (semantics: marlin/vec_host.hpp):
//   struct Engine {
//     using Vec = ...;   vzeros vfrom vwrite vclone vresize vlen vget vset vmul vadd vsub vadd_scaled vscale
//                        vlin vadd_offset veval vdiv_vanishing vdiv_linear vbatch_inverse vshift_down vdomain
//                        vrand vwitness_evals
//     void  vntt(Vec& v, uint32_t log_n, bool inverse, bool coset);            // size 2^log_n, in place
//     // sparse matrices in CSR form, as opaque handles
//     void* csr_upload_filled(const std::vector<uint32_t>& start, Fill fill);  // fill(col, coef) writes the entries
//     IndexOut index_arith(void* a, void* b, void* c, size_t ncons, size_t nvar, size_t ninst, const Domain& H);
//     Vec   vspmv(const void* m, const Vec& x, size_t nout, const Fr* weights);
//     void  csr_free(void* m);
//     void* bases_from_powers(const G1Point& g, const Fr& beta, size_t n);     // resident beta^i * g
//     void  export_bases(void* h, size_t offset, size_t n, G1Point* out);
//     void  free_bases(void* h);
//     void  bases_tune(void* h, size_t typical_n);   // optional restructuring for MSMs of about typical_n scalars
//     size_t msm_submit(void* h, size_t offset, const Vec& scalars, size_t n);   // queue an MSM (scalars stay alive)
//     G1Point msm_result(size_t id);  void msm_drain();
//     size_t msm_local_count(size_t n);   // how many of n scalars this engine processes (its share when sharded)
//   };
// The CUDA engine also has bases_load, csr_download and msm_abandon, which only marlin_abi.cu calls.
//
// Verification is the pairing check of kzg10::batch_check on the host (marlin/pairing.hpp): the two
// opening equations are folded with a verifier-side random scalar into one pairing-product test
// e(sum r_i (C_i - v_i g - v'_i gamma_g + z_i W_i), h) * e(-sum r_i W_i, beta h) == 1.
#pragma once
#include <algorithm>
#include <array>
#include <map>
#include <memory>
#include <stdexcept>
#include <string>

#include "curve_host.hpp"
#include "pairing.hpp"
#include "poly.hpp"
#include "r1cs.hpp"
#include "rng.hpp"

namespace swb {
namespace marlin {

struct MarlinError : std::runtime_error {
    using std::runtime_error::runtime_error;
};

// ------------------------------------------------------------------------------------------------
// sizes (AHPForR1CS::max_degree, SURVEY A.6)
// ------------------------------------------------------------------------------------------------
inline size_t next_pow2(size_t v) {
    size_t p = 1;
    while (p < v) p <<= 1;
    return p;
}
inline size_t ahp_max_degree(size_t num_constraints, size_t num_variables, size_t num_non_zero) {
    const size_t h = next_pow2(std::max(num_constraints, num_variables)), k = next_pow2(num_non_zero), zk = 1;
    return std::max(std::max(2 * h + zk - 2, 3 * h + 2 * zk - 3), std::max(h, 3 * k - 3));
}

// ------------------------------------------------------------------------------------------------
// KZG10 / MarlinKZG10 (SURVEY A.7)
// ------------------------------------------------------------------------------------------------
template <class Engine>
struct UniversalSrs {
    Engine* eng = nullptr;
    size_t max_degree = 0;
    void* powers_of_g = nullptr;              // resident beta^i * g, i <= max_degree
    std::vector<G1Point> powers_of_gamma_g;   // beta^i * gamma_g, i <= hiding_bound + 1 (the only ones trim keeps)
    G1Point g, gamma_g;
    G2Point h, beta_h;                        // verifier side (the trapdoor beta itself is dropped after setup)
    // commit/open traffic over powers_of_g; once an SRS has served a proof's worth of MSMs the engine
    // may restructure the bases for them (window tables on the CUDA engine), see kzg_msm
    mutable size_t msm_calls = 0, msm_points = 0;
    mutable bool tuned = false;
    // number of MSMs after which the engine tunes the bases (0 = never).  Building the window tables
    // costs about as much as 4 proofs and saves ~13 % of each later one, so the default (400 MSMs, some
    // twenty proofs) leaves one-shot and short-lived provers alone and lets a proving service reach the
    // faster path by itself.  SWB_MARLIN_TABLES overrides the default, swb_srs_set_tune_after one SRS.
    long tune_after = [] {
        const char* e = getenv("SWB_MARLIN_TABLES");
        return e ? atol(e) : 400L;
    }();
    ~UniversalSrs() {
        if (eng && powers_of_g) eng->free_bases(powers_of_g);
    }
};

struct Commitment {
    G1Point comm = G1Point::identity();
    bool has_shifted = false;
    G1Point shifted = G1Point::identity();
};
struct Randomness {
    Poly blind;              // hiding polynomial (empty = not hiding)
    Poly shifted_blind;
};
template <class Engine>
struct LabeledPoly {
    std::string label;
    typename Engine::Vec poly;
    bool has_bound = false;
    size_t bound = 0;
    bool hiding = false;
};

template <class Engine>
struct CommitterKey {
    const UniversalSrs<Engine>* srs = nullptr;
    size_t supported_degree = 0;
};

inline Poly rand_poly(size_t degree, ChaChaRng& rng) {   // DensePolynomial::rand: degree + 1 coefficients
    Poly p(degree + 1);
    if (degree < 64) for (auto& c : p) c = rand_fr(rng);
    else rand_fr_bulk(rng, p.data(), p.size());
    return p;
}

// queue the MSM of polynomial p against powers_of_g[offset ..]; the result is fetched with
// srs.eng->msm_result(id).  p must stay alive until then.
template <class Engine>
size_t kzg_msm_submit(const CommitterKey<Engine>& ck, size_t offset, const typename Engine::Vec& p) {
    const UniversalSrs<Engine>& srs = *ck.srs;
    const size_t n = srs.eng->vlen(p);
    if (offset + n > srs.max_degree + 1) throw MarlinError("polynomial degree exceeds the SRS");
    if (!srs.tuned && srs.tune_after > 0 && (long)srs.msm_calls >= srs.tune_after) {
        srs.tuned = true;
        srs.eng->msm_drain();                 // the tables replace the bases other MSMs may still be reading
        ScopedPhase ph("bases_tune");
        srs.eng->bases_tune(srs.powers_of_g, srs.msm_points / srs.msm_calls);
    }
    srs.msm_calls++;
    srs.msm_points += srs.eng->msm_local_count(n);     // what this engine will really process (a share, when sharded)
    ScopedPhase ph("msm");
    return srs.eng->msm_submit(srs.powers_of_g, offset, p, n);
}
template <class Engine>
G1Point kzg_msm_result(const CommitterKey<Engine>& ck, size_t id) {
    ScopedPhase ph("msm");
    return ck.srs->eng->msm_result(id);
}
inline G1Point gamma_msm(const std::vector<G1Point>& gamma, const Poly& blind) {
    G1Xyzz acc = G1Xyzz::identity();
    if (blind.size() > gamma.size()) throw MarlinError("hiding polynomial longer than powers_of_gamma_g");
    for (size_t i = 0; i < blind.size(); i++) {
        G1Point t = g1_mul_fr(gamma[i], blind[i]);
        if (!t.infinity) acc.add_affine(t.x, t.y);
    }
    return to_affine(acc);
}

// MarlinKZG10::commit: per polynomial [commitment][shifted commitment], blinders drawn in that order
template <class Engine>
void pc_commit(const CommitterKey<Engine>& ck, const std::vector<LabeledPoly<Engine>>& polys, ChaChaRng* rng,
               std::vector<Commitment>* comms, std::vector<Randomness>* rands) {
    // all MSMs of the list are queued first (they are independent), blinders are drawn in upstream's
    // order meanwhile, then the results are collected
    struct Pending { size_t comm_id = 0, shifted_id = 0; };
    std::vector<Pending> pend;
    const size_t first = rands->size();
    for (const auto& lp : polys) {
        Randomness r;
        Pending pd;
        if (ck.srs->eng->vlen(lp.poly) > ck.supported_degree + 1) throw MarlinError("polynomial " + lp.label + " too large for the committer key");
        pd.comm_id = kzg_msm_submit(ck, 0, lp.poly);
        if (lp.hiding) r.blind = rand_poly(2, *rng);     // hiding_bound + 1 = degree 2
        if (lp.has_bound) {
            pd.shifted_id = kzg_msm_submit(ck, ck.srs->max_degree - lp.bound, lp.poly);
            if (lp.hiding) r.shifted_blind = rand_poly(2, *rng);
        }
        pend.push_back(pd);
        rands->push_back(r);
    }
    for (size_t i = 0; i < polys.size(); i++) {
        const auto& lp = polys[i];
        const Randomness& r = (*rands)[first + i];
        Commitment c;
        c.comm = kzg_msm_result(ck, pend[i].comm_id);
        if (lp.hiding) c.comm = g1_add(c.comm, gamma_msm(ck.srs->powers_of_gamma_g, r.blind));
        if (lp.has_bound) {
            c.has_shifted = true;
            c.shifted = kzg_msm_result(ck, pend[i].shifted_id);
            if (lp.hiding) c.shifted = g1_add(c.shifted, gamma_msm(ck.srs->powers_of_gamma_g, r.shifted_blind));
        }
        comms->push_back(c);
    }
}

struct PcProof {
    G1Point w = G1Point::identity();
    bool has_random_v = false;
    Fr random_v = Fr::zero();
};

// MarlinKZG10::open at one point for a list of polynomials (opening challenge powers xi^j, one per
// polynomial and one more for a shifted part)
template <class Engine>
PcProof pc_open(const CommitterKey<Engine>& ck, const std::vector<const LabeledPoly<Engine>*>& polys,
                const std::vector<const Randomness*>& rands, const Fr& point, const Fr& xi) {
    using Vec = typename Engine::Vec;
    Engine& eng = *ck.srs->eng;
    Vec p = eng.vzeros(0);
    Poly r, shifted_r_witness;
    bool hiding = false;
    Fr shifted_r_value = Fr::zero();
    Fr chal = Fr::one();
    // shifted witnesses are committed against different offsets of the powers, so they are
    // accumulated per offset
    std::map<size_t, Vec> shifted_by_offset;
    for (size_t j = 0; j < polys.size(); j++) {
        eng.vadd_scaled(p, chal, polys[j]->poly);
        if (!rands[j]->blind.empty()) { poly_add_scaled(r, chal, rands[j]->blind); hiding = true; }
        chal = chal * xi;
        if (polys[j]->has_bound) {
            Vec wj = eng.vdiv_linear(polys[j]->poly, point);
            const size_t off = ck.srs->max_degree - polys[j]->bound;
            auto it = shifted_by_offset.find(off);
            if (it == shifted_by_offset.end()) it = shifted_by_offset.emplace(off, eng.vzeros(0)).first;
            eng.vadd_scaled(it->second, chal, wj);
            if (!rands[j]->shifted_blind.empty()) {
                hiding = true;
                Poly rw = poly_divide_by_linear(rands[j]->shifted_blind, point);
                poly_add_scaled(shifted_r_witness, chal, rw);
                shifted_r_value = shifted_r_value + chal * poly_eval(rands[j]->shifted_blind, point);
            }
            chal = chal * xi;
        }
    }
    PcProof pr;
    Vec witness = eng.vdiv_linear(p, point);
    const size_t wit_id = kzg_msm_submit(ck, 0, witness);
    std::vector<size_t> shifted_ids;
    for (auto& kv : shifted_by_offset) shifted_ids.push_back(kzg_msm_submit(ck, kv.first, kv.second));
    G1Xyzz w = to_xyzz(kzg_msm_result(ck, wit_id));
    if (hiding) {
        Poly rwit = poly_divide_by_linear(r, point);
        G1Point t = gamma_msm(ck.srs->powers_of_gamma_g, rwit);
        if (!t.infinity) w.add_affine(t.x, t.y);
        pr.has_random_v = true;
        pr.random_v = poly_eval(r, point);
    }
    for (size_t id : shifted_ids) {
        G1Point t = kzg_msm_result(ck, id);
        if (!t.infinity) w.add_affine(t.x, t.y);
    }
    if (!shifted_r_witness.empty()) {
        G1Point t = gamma_msm(ck.srs->powers_of_gamma_g, shifted_r_witness);
        if (!t.infinity) w.add_affine(t.x, t.y);
        pr.random_v = pr.random_v + shifted_r_value;
    }
    pr.w = to_affine(w);
    return pr;
}

// ------------------------------------------------------------------------------------------------
// index (AHPForR1CS::index + MarlinKZG10::trim/commit; SURVEY A.8, joint arithmetisation)
// ------------------------------------------------------------------------------------------------
struct IndexInfo {
    size_t num_variables = 0, num_constraints = 0, num_non_zero = 0, num_instance = 0;
};

template <class Engine>
struct ProvingKey {
    IndexInfo info;
    Domain dom_h, dom_k, dom_x;
    std::vector<LabeledPoly<Engine>> index_polys;   // row, col, a_val, b_val, c_val, row_col (resident)
    typename Engine::Vec row_evals, col_evals, val_a_evals, val_b_evals, val_c_evals;   // on K (resident)
    std::vector<Commitment> index_comms;
    CommitterKey<Engine> ck;        // ck.srs->eng is the engine of every operation on the key; the SRS outlives the key
    // the matrices where the engine keeps its vectors (device memory for the CUDA engine): A, B, C in CSR over
    // z = (instance | witness), and the entries of all three regrouped by the H position of their column, tagged by
    // matrix (for t = sum_M eta_M M^T r_alpha)
    void *m_a = nullptr, *m_b = nullptr, *m_c = nullptr, *m_t = nullptr;
    ProvingKey() {}
    ProvingKey(const ProvingKey&) = delete;
    ProvingKey& operator=(const ProvingKey&) = delete;
    ~ProvingKey() {
        if (!ck.srs) return;
        void* ms[4] = {m_a, m_b, m_c, m_t};
        for (void* m : ms)
            if (m) ck.srs->eng->csr_free(m);
    }
};
// IndexVerifierKey: index info + index commitments + MarlinKZG10's VerifierKey (g, gamma_g, h, beta_h,
// degree_bounds_and_shift_powers); self-contained, independent of the engine
struct VerifyingKey {
    IndexInfo info;
    std::vector<Commitment> index_comms;
    G1Point g, gamma_g;
    G2Point h, beta_h;
    size_t max_degree = 0;
    std::vector<std::pair<size_t, G1Point>> shift_powers;   // (bound, beta^(D - bound) g)
    const G1Point* shift_power(size_t bound) const {
        for (auto& sp : shift_powers)
            if (sp.first == bound) return &sp.second;
        return nullptr;
    }
    // serialize_verifying_key / deserialize_verifying_key (reference src/marlin/serialization.rs:19-31):
    // index_info (4 x u64), index_comms, then MarlinKZG10's VerifierKey -- g, gamma_g (48 B), h, beta_h
    // (96 B), Some(degree_bounds_and_shift_powers), max_degree, supported_degree -- in ark-serialize's
    // compressed conventions.  Layout follows SURVEY row a7; unpinned against real arkworks bytes.
    std::vector<uint8_t> serialize() const;
    static bool deserialize(const uint8_t* p, size_t len, VerifyingKey* out);
};

inline void put_commitment_canonical(std::vector<uint8_t>& out, const Commitment& c) {
    put_g1_compressed(out, c.comm);
    out.push_back(c.has_shifted ? 1 : 0);
    if (c.has_shifted) put_g1_compressed(out, c.shifted);
}
inline bool get_commitment_canonical(const uint8_t*& p, const uint8_t* end, Commitment* c) {
    if (!get_g1_compressed(p, end, &c->comm) || p >= end) return false;
    c->has_shifted = *p++ != 0;
    return !c->has_shifted || get_g1_compressed(p, end, &c->shifted);
}
inline std::vector<uint8_t> VerifyingKey::serialize() const {
    std::vector<uint8_t> out;
    put_u64(out, info.num_variables);
    put_u64(out, info.num_constraints);
    put_u64(out, info.num_non_zero);
    put_u64(out, info.num_instance);
    put_u64(out, index_comms.size());
    for (auto& c : index_comms) put_commitment_canonical(out, c);
    put_g1_compressed(out, g);
    put_g1_compressed(out, gamma_g);
    put_g2_compressed(out, h);
    put_g2_compressed(out, beta_h);
    out.push_back(1);                                   // Option::Some
    put_u64(out, shift_powers.size());
    for (auto& sp : shift_powers) {
        put_u64(out, sp.first);
        put_g1_compressed(out, sp.second);
    }
    put_u64(out, max_degree);
    put_u64(out, ahp_max_degree(info.num_constraints, info.num_variables, info.num_non_zero));
    return out;
}
inline bool VerifyingKey::deserialize(const uint8_t* p, size_t len, VerifyingKey* out) {
    const uint8_t* end = p + len;
    uint64_t v[4], n;
    for (int i = 0; i < 4; i++)
        if (!get_u64(p, end, &v[i])) return false;
    // sizes a verifier would turn into evaluation domains: refuse what no radix-2 domain of Fr can hold
    for (int i = 0; i < 4; i++)
        if (v[i] > ((uint64_t)1 << SWB_FR_TWO_ADICITY)) return false;
    if (v[3] == 0 || v[3] > v[0]) return false;
    out->info = IndexInfo{(size_t)v[0], (size_t)v[1], (size_t)v[2], (size_t)v[3]};
    if (!get_u64(p, end, &n) || n > 64) return false;
    out->index_comms.resize(n);
    for (auto& c : out->index_comms)
        if (!get_commitment_canonical(p, end, &c)) return false;
    if (!get_g1_compressed(p, end, &out->g) || !get_g1_compressed(p, end, &out->gamma_g)) return false;
    if (!get_g2_compressed(p, end, &out->h) || !get_g2_compressed(p, end, &out->beta_h)) return false;
    if (p >= end || *p++ != 1) return false;
    if (!get_u64(p, end, &n) || n > 64) return false;
    out->shift_powers.resize(n);
    for (auto& sp : out->shift_powers) {
        uint64_t b;
        if (!get_u64(p, end, &b) || !get_g1_compressed(p, end, &sp.second)) return false;
        sp.first = (size_t)b;
    }
    uint64_t md, sd;
    if (!get_u64(p, end, &md) || !get_u64(p, end, &sd)) return false;
    out->max_degree = (size_t)md;
    return p == end;
}

inline void put_commitment_bytes(std::vector<uint8_t>& out, const Commitment& c) {   // ToBytes, 195 B
    put_g1_uncompressed(out, c.comm);
    out.push_back(c.has_shifted ? 1 : 0);
    put_g1_uncompressed(out, c.has_shifted ? c.shifted : G1Point::identity());
}
inline void put_vk_bytes(std::vector<uint8_t>& out, const IndexInfo& info, const std::vector<Commitment>& comms) {
    put_u64(out, info.num_variables);
    put_u64(out, info.num_constraints);
    put_u64(out, info.num_non_zero);
    for (auto& c : comms) put_commitment_bytes(out, c);
}

template <class Engine>
std::unique_ptr<UniversalSrs<Engine>> universal_setup(Engine& eng, size_t num_constraints, size_t num_variables,
                                                      size_t num_non_zero, ChaChaRng& rng) {
    auto srs = std::make_unique<UniversalSrs<Engine>>();
    srs->eng = &eng;
    srs->max_degree = ahp_max_degree(num_constraints, num_variables, num_non_zero);
    // KZG10::setup draw order: beta, g, gamma_g, h (G2)
    const Fr beta = rand_fr(rng);
    srs->g = g1_rand(rng);
    srs->gamma_g = g1_rand(rng);
    srs->h = g2_rand(rng);
    srs->beta_h = g2_mul_fr(srs->h, beta);
    srs->powers_of_g = eng.bases_from_powers(srs->g, beta, srs->max_degree + 1);
    // upstream also tabulates all max_degree + 2 powers of gamma_g; only the first
    // hiding_bound + 2 = 3 survive trim, so only those are materialised here
    srs->powers_of_gamma_g.resize(3);
    Fr bp = Fr::one();
    for (int i = 0; i < 3; i++) {
        srs->powers_of_gamma_g[i] = g1_mul_fr(srs->gamma_g, bp);
        bp = bp * beta;
    }
    return srs;
}

template <class Engine>
void index(const UniversalSrs<Engine>& srs, const R1cs& cs, ProvingKey<Engine>* pk, VerifyingKey* vk) {
    Engine& eng = *srs.eng;
    ScopedPhase ph_total("total");
    std::unique_ptr<ScopedPhase> ph(new ScopedPhase("i0_pad"));
    // pad_input_for_indexer_and_prover + make_matrices_square without copying the matrices: the instance
    // count goes up to a power of two (witness columns shift by `shift`), then either empty constraints
    // or dummy witnesses make the system square
    size_t ninst = 1;
    while (ninst < cs.num_instance) ninst <<= 1;
    const uint32_t shift = (uint32_t)(ninst - cs.num_instance);
    const size_t orig_inst = cs.num_instance;
    auto col_of = [&](uint32_t c) { return c >= orig_inst ? c + shift : c; };
    const size_t nrows_real = cs.a.size();
    const size_t nvar = std::max(ninst + cs.num_witness, nrows_real), ncons = nvar;
    static const SparseRow empty_row;
    auto row_of = [&](const std::vector<SparseRow>& m, size_t r) -> const SparseRow& { return r < nrows_real ? m[r] : empty_row; };
    pk->dom_h = Domain(ncons);
    pk->dom_x = Domain(ninst);
    const Domain& H = pk->dom_h;
    // The engine arithmetises where its vectors live (index_ops.cu on the CUDA engine): here the three matrices are
    // only flattened into CSR arrays and staged there -- they are needed there anyway, for z_A, z_B, z_C.
    ph.reset(); ph.reset(new ScopedPhase("i4_upload"));
    pk->ck.srs = &srs;             // from here on the key frees its matrices through srs.eng, also when index throws
    auto stage_rows = [&](const std::vector<SparseRow>& m) {
        std::vector<uint32_t> start(ncons + 1, 0);
        for (size_t r = 0; r < ncons; r++) start[r + 1] = start[r] + (uint32_t)row_of(m, r).e.size();
        return eng.csr_upload_filled(start, [&](uint32_t* col, Fr* coef) {
#pragma omp parallel for schedule(static)
            for (size_t r = 0; r < m.size(); r++) {
                uint32_t at = start[r];
                for (auto& e : m[r].e) { col[at] = col_of(e.second); coef[at] = e.first; at++; }
            }
        });
    };
    pk->m_a = stage_rows(cs.a);
    pk->m_b = stage_rows(cs.b);
    pk->m_c = stage_rows(cs.c);
    ph.reset(); ph.reset(new ScopedPhase("i2_arith"));
    auto out = eng.index_arith(pk->m_a, pk->m_b, pk->m_c, ncons, nvar, ninst, H);
    pk->m_t = out.m_t;
    const size_t nnz = out.nnz;
    pk->info = IndexInfo{nvar, ncons, nnz, ninst};
    pk->dom_k = Domain(nnz);
    if (ahp_max_degree(pk->info.num_constraints, nvar, nnz) > srs.max_degree)
        throw MarlinError("index: circuit exceeds the universal SRS bound");
    pk->row_evals = std::move(out.row); pk->col_evals = std::move(out.col);
    pk->val_a_evals = std::move(out.va); pk->val_b_evals = std::move(out.vb); pk->val_c_evals = std::move(out.vc);
    ph.reset(); ph.reset(new ScopedPhase("i5_polys_commit"));
    const char* names[6] = {"row", "col", "a_val", "b_val", "c_val", "row_col"};
    const Domain& K = pk->dom_k;
    const typename Engine::Vec* evs[6] = {&pk->row_evals, &pk->col_evals, &pk->val_a_evals, &pk->val_b_evals, &pk->val_c_evals, &out.rowcol};
    pk->index_polys.clear();
    for (int i = 0; i < 6; i++) {
        LabeledPoly<Engine> lp;
        lp.label = names[i];
        lp.poly = eng.vclone(*evs[i]);
        eng.vntt(lp.poly, K.log_n, true, false);
        pk->index_polys.push_back(std::move(lp));
    }
    pk->ck.supported_degree = ahp_max_degree(pk->info.num_constraints, nvar, nnz);
    std::vector<Randomness> unused;
    pk->index_comms.clear();
    pc_commit(pk->ck, pk->index_polys, nullptr, &pk->index_comms, &unused);
    vk->info = pk->info;
    vk->index_comms = pk->index_comms;
    vk->g = srs.g;
    vk->gamma_g = srs.gamma_g;
    vk->h = srs.h;
    vk->beta_h = srs.beta_h;
    vk->max_degree = srs.max_degree;
    vk->shift_powers.clear();
    // get_degree_bounds: |H| - 2, |K| - 2; marlin_pc::trim sorts and dedups the enforced bounds
    std::vector<size_t> bounds = {H.n - 2, K.n - 2};
    std::sort(bounds.begin(), bounds.end());
    bounds.erase(std::unique(bounds.begin(), bounds.end()), bounds.end());
    for (size_t bound : bounds) {
        G1Point sp;
        eng.export_bases(srs.powers_of_g, srs.max_degree - bound, 1, &sp);
        vk->shift_powers.push_back({bound, sp});
    }
}

// ------------------------------------------------------------------------------------------------
// proof
// ------------------------------------------------------------------------------------------------
struct Proof {
    std::vector<std::vector<Commitment>> commitments;   // [w,z_a,z_b,mask] [t,g_1,h_1] [g_2,h_2]
    std::vector<Fr> evaluations;                        // g_1(beta), g_2(gamma), t(beta), z_b(beta)
    std::vector<PcProof> pc_proofs;                     // @beta, @gamma

    // ark-serialize CanonicalSerialize (SURVEY row a7, A.9)
    std::vector<uint8_t> serialize() const {
        std::vector<uint8_t> out;
        put_u64(out, commitments.size());
        for (auto& round : commitments) {
            put_u64(out, round.size());
            for (auto& c : round) {
                put_g1_compressed(out, c.comm);
                out.push_back(c.has_shifted ? 1 : 0);
                if (c.has_shifted) put_g1_compressed(out, c.shifted);
            }
        }
        put_u64(out, evaluations.size());
        for (auto& e : evaluations) put_fr_canonical(out, e);
        put_u64(out, 3);                       // prover_messages: three EmptyMessage = Option::None
        for (int i = 0; i < 3; i++) out.push_back(0);
        put_u64(out, pc_proofs.size());
        for (auto& p : pc_proofs) {
            put_g1_compressed(out, p.w);
            out.push_back(p.has_random_v ? 1 : 0);
            if (p.has_random_v) put_fr_canonical(out, p.random_v);
        }
        out.push_back(0);                      // BatchLCProof.evals: None
        return out;
    }
    static bool deserialize(const uint8_t* p, size_t len, Proof* out) { return deserialize(p, len, out, get_g1_compressed); }
    // The same parser with the G1 points read by `get_point(p, end, G1Point* out)`, which has the signature and contract of
    // get_g1_compressed: the batch verifier collects the encodings here and decodes them all at once on the GPU.
    template <class PointReader>
    static bool deserialize(const uint8_t* p, size_t len, Proof* out, PointReader&& get_point) {
        const uint8_t* end = p + len;
        auto get_u64 = [&](uint64_t* v) {
            if (end - p < 8) return false;
            *v = 0;
            for (int b = 0; b < 8; b++) *v |= (uint64_t)p[b] << (8 * b);
            p += 8;
            return true;
        };
        uint64_t n;
        if (!get_u64(&n) || n > 8) return false;
        out->commitments.assign(n, {});
        for (auto& round : out->commitments) {
            uint64_t m;
            if (!get_u64(&m) || m > 64) return false;
            round.resize(m);
            for (auto& c : round) {
                if (!get_point(p, end, &c.comm)) return false;
                if (p >= end) return false;
                c.has_shifted = *p++ != 0;
                if (c.has_shifted && !get_point(p, end, &c.shifted)) return false;
            }
        }
        if (!get_u64(&n) || n > 64) return false;
        out->evaluations.resize(n);
        for (auto& e : out->evaluations)
            if (!get_fr_canonical(p, end, &e)) return false;
        if (!get_u64(&n) || n != 3 || end - p < 3) return false;
        p += 3;
        if (!get_u64(&n) || n > 8) return false;
        out->pc_proofs.resize(n);
        for (auto& pr : out->pc_proofs) {
            if (!get_point(p, end, &pr.w)) return false;
            if (p >= end) return false;
            pr.has_random_v = *p++ != 0;
            if (pr.has_random_v && !get_fr_canonical(p, end, &pr.random_v)) return false;
        }
        return end - p == 1 && *p == 0;
    }
};

// ------------------------------------------------------------------------------------------------
// transcript helpers shared by prover and verifier
// ------------------------------------------------------------------------------------------------
inline Fr sample_outside(const Domain& d, ChaChaRng& rng) {     // sample_element_outside_domain
    Fr t = rand_fr(rng);
    while (d.vanishing_at(t).is_zero()) t = rand_fr(rng);
    return t;
}
inline Fr fr_from_u128(const uint64_t w[2]) {
    Fr c = Fr::zero();
    c.l[0] = (uint32_t)w[0]; c.l[1] = (uint32_t)(w[0] >> 32);
    c.l[2] = (uint32_t)w[1]; c.l[3] = (uint32_t)(w[1] >> 32);
    return c.from_canonical();
}
inline std::vector<uint8_t> round_bytes(const std::vector<Commitment>& comms) {
    std::vector<uint8_t> out;
    for (auto& c : comms) put_commitment_bytes(out, c);
    return out;                                   // the prover message is EmptyMessage: no bytes
}
struct Challenges {
    Fr alpha, eta_a, eta_b, eta_c, beta, gamma, xi;
};
// a linear combination of committed polynomials plus a constant; the constant moves to the claimed
// value (poly-commit's handling of LCTerm::One): sum coeff_i p_i(z) must equal -constant
struct LinComb {
    std::string label;
    std::vector<std::pair<Fr, std::string>> terms;
    Fr constant = Fr::zero();
};
struct LcInputs {
    Fr g1_beta, g2_gamma, t_beta, zb_beta;       // reported evaluations
    Fr x_hat_beta, v_x_beta;                     // from the public input
};
inline void build_lcs(const Domain& H, const Domain& K, const Challenges& ch, const LcInputs& in, LinComb* outer, LinComb* inner) {
    const Fr vh_a = H.vanishing_at(ch.alpha), vh_b = H.vanishing_at(ch.beta), vk_g = K.vanishing_at(ch.gamma);
    const Fr r_ab = H.bivariate(ch.alpha, ch.beta);
    // outer: mask + r(a,b)(eta_a + eta_c z_b(b)) z_a + r(a,b) eta_b z_b(b) - t(b) v_X(b) w - t(b) x^(b)
    //        - v_H(b) h_1 - b g_1(b) = 0
    outer->label = "outer_sumcheck";
    outer->terms = {{Fr::one(), "mask_poly"},
                    {r_ab * (ch.eta_a + ch.eta_c * in.zb_beta), "z_a"},
                    {(in.t_beta * in.v_x_beta).neg(), "w"},
                    {vh_b.neg(), "h_1"}};
    outer->constant = r_ab * ch.eta_b * in.zb_beta - in.t_beta * in.x_hat_beta - ch.beta * in.g1_beta;
    // inner: v_H(a) v_H(b) (eta_a a_val + eta_b b_val + eta_c c_val)
    //        - (ab - a row - b col + row_col)(g g_2(g) + t(b)/|K|) - v_K(g) h_2 = 0
    const Fr s = ch.gamma * in.g2_gamma + in.t_beta * K.size_inv;
    const Fr vv = vh_a * vh_b;
    inner->label = "inner_sumcheck";
    inner->terms = {{vv * ch.eta_a, "a_val"}, {vv * ch.eta_b, "b_val"}, {vv * ch.eta_c, "c_val"},
                    {ch.alpha * s, "row"}, {ch.beta * s, "col"}, {s.neg(), "row_col"}, {vk_g.neg(), "h_2"}};
    inner->constant = (ch.alpha * ch.beta * s).neg();
}

// ------------------------------------------------------------------------------------------------
// prove (AHPForR1CS prover rounds + MarlinKZG10 commit/open; SURVEY A.9)
// ------------------------------------------------------------------------------------------------
template <class Engine>
Proof prove(const ProvingKey<Engine>& pk, const R1cs& cs, ChaChaRng& zk_rng) {
    Engine& eng = *pk.ck.srs->eng;
    if (!cs.has_assignment) throw MarlinError("prove: constraint system has no assignment");
    // the assignment after pad_input_for_indexer_and_prover + make_matrices_square (the matrices
    // themselves live in the proving key): instance padded with zeros to a power of two, dummy
    // witnesses of value one when there are more constraints than variables
    std::vector<Fr> instance = cs.instance;                // small; the witness is used where it lies
    size_t dummy_witnesses = 0;
    {
        size_t target = 1;
        while (target < instance.size()) target <<= 1;
        instance.resize(target, Fr::zero());
        size_t nv = instance.size() + cs.witness.size(), nc = cs.num_constraints();
        if (nc < nv) nc = nv;
        else if (nv < nc) { dummy_witnesses = nc - nv; nv = nc; }
        if (nv != pk.info.num_variables || nc != pk.info.num_constraints || instance.size() != pk.info.num_instance)
            throw MarlinError("prove: constraint system does not match the proving key");
    }
    using Vec = typename Engine::Vec;
    const Domain &H = pk.dom_h, &K = pk.dom_k, &X = pk.dom_x;
    const size_t nh = H.n, nx = X.n, ratio = nh / nx;
    auto ntt = [&](Vec& v, const Domain& d, bool inverse) {
        eng.vresize(v, d.n);
        ScopedPhase ph("ntt");
        eng.vntt(v, d.log_n, inverse, false);
    };
    auto poly_mul = [&](const Vec& a, const Vec& b) {
        const size_t la = eng.vlen(a), lb = eng.vlen(b);
        Domain d(la + lb - 1);
        Vec ea = eng.vclone(a), eb = eng.vclone(b);
        ntt(ea, d, false);
        ntt(eb, d, false);
        eng.vmul(ea, eb);
        ntt(ea, d, true);
        return ea;
    };
    ScopedPhase ph_total("total");
    std::unique_ptr<ScopedPhase> ph(new ScopedPhase("r0_init"));
    // ---- init: z_A = A z, z_B = B z on the engine (prover_init) ------------------------------------
    Vec z_vec;
    {
        // z = (instance | witness | dummy witnesses = 1): uploaded part by part, no concatenated host copy
        const size_t ni = instance.size(), nw = cs.witness.size();
        z_vec = eng.vzeros(ni + nw + dummy_witnesses);
        eng.vwrite(z_vec, 0, instance.data(), ni);
        eng.vwrite(z_vec, ni, cs.witness.data(), nw);
        if (dummy_witnesses) {
            const std::vector<Fr> ones(dummy_witnesses, Fr::one());
            eng.vwrite(z_vec, ni + nw, ones.data(), dummy_witnesses);
        }
    }
    Vec za_ev = eng.vspmv(pk.m_a, z_vec, nh, nullptr), zb_ev = eng.vspmv(pk.m_b, z_vec, nh, nullptr);
    {
        Vec chk = eng.vspmv(pk.m_c, z_vec, nh, nullptr);
        Vec prod = eng.vclone(za_ev);
        eng.vmul(prod, zb_ev);
        eng.vsub(chk, prod);
        if (eng.vlen(chk) != 0) throw MarlinError("prove: constraint system is not satisfied");
    }
    std::vector<Fr> public_input(instance.begin() + 1, instance.end());   // padded, without the one
    FiatShamirRng fs;
    {
        std::vector<uint8_t> init;
        const char* name = "MARLIN-2019";
        init.insert(init.end(), name, name + 11);
        put_vk_bytes(init, pk.info, pk.index_comms);
        for (auto& x : public_input) put_fr_canonical(init, x);
        fs.initialize(init);
    }
    // ---- round 1 ---------------------------------------------------------------------------------
    ph.reset(); ph.reset(new ScopedPhase("r1_polys"));
    Vec x_hat = eng.vfrom(instance);
    ntt(x_hat, X, true);
    Vec w_poly;
    const Fr rho_w = rand_fr(zk_rng);
    {
        ScopedPhase sp("r1_polys.w");
        // w on H: 0 on the X-subdomain, witness - x^ elsewhere
        Vec xh_on_h = eng.vclone(x_hat);
        ntt(xh_on_h, H, false);
        Vec w_ev = eng.vwitness_evals(z_vec, instance.size(), xh_on_h, ratio);
        ntt(w_ev, H, true);
        // + rho_w * (X^nh - 1), then / v_X
        eng.vresize(w_ev, nh + 1);
        eng.vset(w_ev, 0, eng.vget(w_ev, 0) - rho_w);
        eng.vset(w_ev, nh, rho_w);
        Vec rem;
        eng.vdiv_vanishing(w_ev, nx, &w_poly, &rem);
    }
    auto blinded_interp = [&](Vec& ev, const Fr& rho) {
        Vec p = std::move(ev);
        ntt(p, H, true);
        eng.vresize(p, nh + 1);
        eng.vset(p, 0, eng.vget(p, 0) - rho);
        eng.vset(p, nh, rho);
        return p;
    };
    const Fr rho_a = rand_fr(zk_rng);
    Vec za_poly, zb_poly;
    {
        ScopedPhase sp("r1_polys.z");
        za_poly = blinded_interp(za_ev, rho_a);
    }
    const Fr rho_b = rand_fr(zk_rng);
    {
        ScopedPhase sp("r1_polys.z");
        zb_poly = blinded_interp(zb_ev, rho_b);
    }
    Vec mask;
    {
        ScopedPhase sp("r1_polys.mask");
        mask = eng.vrand(zk_rng, 3 * nh);                      // degree 3|H| + 2 zk - 3
        Fr r0 = Fr::zero();
        for (size_t i = 0; i < 3 * nh; i += nh) r0 = r0 + eng.vget(mask, i);
        eng.vset(mask, 0, eng.vget(mask, 0) - r0);             // sum over H becomes zero
    }
    std::vector<LabeledPoly<Engine>> first(4);
    first[0].label = "w"; first[0].poly = std::move(w_poly); first[0].hiding = true;
    first[1].label = "z_a"; first[1].poly = std::move(za_poly); first[1].hiding = true;
    first[2].label = "z_b"; first[2].poly = std::move(zb_poly); first[2].hiding = true;
    first[3].label = "mask_poly"; first[3].poly = std::move(mask);
    const Vec &w_p = first[0].poly, &za_p = first[1].poly, &zb_p = first[2].poly, &mask_p = first[3].poly;
    Proof proof;
    proof.commitments.resize(3);
    std::vector<Randomness> first_r, second_r, third_r;
    ph.reset(); ph.reset(new ScopedPhase("r1_commit"));
    pc_commit(pk.ck, first, &zk_rng, &proof.commitments[0], &first_r);
    ph.reset(); ph.reset(new ScopedPhase("r2_polys"));
    fs.absorb(round_bytes(proof.commitments[0]));
    Challenges ch;
    ch.alpha = sample_outside(H, fs.rng());
    ch.eta_a = rand_fr(fs.rng());
    ch.eta_b = rand_fr(fs.rng());
    ch.eta_c = rand_fr(fs.rng());
    // ---- round 2 ---------------------------------------------------------------------------------
    const Fr vh_alpha = H.vanishing_at(ch.alpha);
    Vec r_alpha = eng.vdomain(H.log_n);                      // r(alpha, h) = v_H(alpha) / (alpha - h)
    eng.vlin(r_alpha, ch.alpha, Fr::one().neg());
    eng.vbatch_inverse(r_alpha);
    eng.vscale(r_alpha, vh_alpha);
    // t on H: t(H[pos(c)]) = sum_M eta_M sum_r M[r][c] r_alpha(H[r])   (sparse transpose product on the engine)
    Vec t_poly;
    {
        ScopedPhase sp("r2_polys.t");
        const Fr etas[3] = {ch.eta_a, ch.eta_b, ch.eta_c};
        t_poly = eng.vspmv(pk.m_t, r_alpha, nh, etas);
    }
    ntt(t_poly, H, true);
    ntt(r_alpha, H, true);                                   // now the polynomial r(alpha, X)
    Vec g1_poly, h1_poly;
    {
        Vec summed = poly_mul(za_p, zb_p);                   // z_c = z_a z_b
        eng.vscale(summed, ch.eta_c);
        eng.vadd_scaled(summed, ch.eta_a, za_p);
        eng.vadd_scaled(summed, ch.eta_b, zb_p);
        Vec z_poly = eng.vclone(x_hat);                      // z = w v_X + x^
        eng.vadd_offset(z_poly, nx, w_p, false);
        eng.vadd_offset(z_poly, 0, w_p, true);
        Vec q1 = poly_mul(r_alpha, summed);
        Vec tz = poly_mul(t_poly, z_poly);
        eng.vsub(q1, tz);
        eng.vadd(q1, mask_p);
        Vec rem;
        eng.vdiv_vanishing(q1, nh, &h1_poly, &rem);
        if (!eng.vget(rem, 0).is_zero()) throw MarlinError("prove: outer sumcheck does not sum to zero");
        g1_poly = eng.vshift_down(rem, 1);                   // rem = X g_1
    }
    std::vector<LabeledPoly<Engine>> second(3);
    second[0].label = "t"; second[0].poly = std::move(t_poly);
    second[1].label = "g_1"; second[1].poly = std::move(g1_poly); second[1].has_bound = true; second[1].bound = nh - 2; second[1].hiding = true;
    second[2].label = "h_1"; second[2].poly = std::move(h1_poly); second[2].hiding = true;
    ph.reset(); ph.reset(new ScopedPhase("r2_commit"));
    pc_commit(pk.ck, second, &zk_rng, &proof.commitments[1], &second_r);
    ph.reset(); ph.reset(new ScopedPhase("r3_polys"));
    fs.absorb(round_bytes(proof.commitments[1]));
    ch.beta = sample_outside(H, fs.rng());
    // ---- round 3 ---------------------------------------------------------------------------------
    const Fr vh_beta = H.vanishing_at(ch.beta), vv = vh_alpha * vh_beta;
    Vec f_poly;
    {
        Vec den = eng.vclone(pk.row_evals);                  // (beta - row)(alpha - col)
        eng.vlin(den, ch.beta, Fr::one().neg());
        Vec d2 = eng.vclone(pk.col_evals);
        eng.vlin(d2, ch.alpha, Fr::one().neg());
        eng.vmul(den, d2);
        eng.vbatch_inverse(den);
        Vec num = eng.vclone(pk.val_a_evals);
        eng.vscale(num, vv * ch.eta_a);
        eng.vadd_scaled(num, vv * ch.eta_b, pk.val_b_evals);
        eng.vadd_scaled(num, vv * ch.eta_c, pk.val_c_evals);
        eng.vmul(num, den);
        f_poly = std::move(num);
    }
    ntt(f_poly, K, true);
    Vec g2_poly = eng.vshift_down(f_poly, 1);
    Vec h2_poly;
    {
        const Vec &row = pk.index_polys[0].poly, &col = pk.index_polys[1].poly, &rc = pk.index_polys[5].poly;
        Vec a_poly = eng.vclone(pk.index_polys[2].poly);
        eng.vscale(a_poly, vv * ch.eta_a);
        eng.vadd_scaled(a_poly, vv * ch.eta_b, pk.index_polys[3].poly);
        eng.vadd_scaled(a_poly, vv * ch.eta_c, pk.index_polys[4].poly);
        Vec b_poly = eng.vclone(rc);
        eng.vadd_scaled(b_poly, ch.alpha.neg(), row);
        eng.vadd_scaled(b_poly, ch.beta.neg(), col);
        eng.vset(b_poly, 0, eng.vget(b_poly, 0) + ch.alpha * ch.beta);
        Vec bf = poly_mul(b_poly, f_poly);
        eng.vsub(a_poly, bf);
        Vec rem;
        eng.vdiv_vanishing(a_poly, K.n, &h2_poly, &rem);
        if (eng.vlen(rem) != 0) throw MarlinError("prove: inner sumcheck identity does not hold on K");
    }
    std::vector<LabeledPoly<Engine>> third(2);
    third[0].label = "g_2"; third[0].poly = std::move(g2_poly); third[0].has_bound = true; third[0].bound = K.n - 2;
    third[1].label = "h_2"; third[1].poly = std::move(h2_poly);
    ph.reset(); ph.reset(new ScopedPhase("r3_commit"));
    pc_commit(pk.ck, third, &zk_rng, &proof.commitments[2], &third_r);
    ph.reset(); ph.reset(new ScopedPhase("r4_evals_lcs"));
    fs.absorb(round_bytes(proof.commitments[2]));
    ch.gamma = rand_fr(fs.rng());
    // ---- evaluations, linear combinations, openings -----------------------------------------------
    LcInputs in;
    in.g1_beta = eng.veval(second[1].poly, ch.beta);
    in.g2_gamma = eng.veval(third[0].poly, ch.gamma);
    in.t_beta = eng.veval(second[0].poly, ch.beta);
    in.zb_beta = eng.veval(zb_p, ch.beta);
    in.x_hat_beta = eng.veval(x_hat, ch.beta);
    in.v_x_beta = X.vanishing_at(ch.beta);
    proof.evaluations = {in.g1_beta, in.g2_gamma, in.t_beta, in.zb_beta};
    {
        std::vector<uint8_t> eb;
        for (auto& e : proof.evaluations) put_fr_canonical(eb, e);
        fs.absorb(eb);
    }
    uint64_t u[2];
    fs.rng().next_u128(u);
    ch.xi = fr_from_u128(u);
    LinComb outer, inner;
    build_lcs(H, K, ch, in, &outer, &inner);
    std::map<std::string, std::pair<const LabeledPoly<Engine>*, const Randomness*>> by_label;
    for (size_t i = 0; i < first.size(); i++) by_label[first[i].label] = {&first[i], &first_r[i]};
    for (size_t i = 0; i < second.size(); i++) by_label[second[i].label] = {&second[i], &second_r[i]};
    for (size_t i = 0; i < third.size(); i++) by_label[third[i].label] = {&third[i], &third_r[i]};
    static const Randomness no_rand;
    for (auto& ip : pk.index_polys) by_label[ip.label] = {&ip, &no_rand};
    auto make_lc = [&](const LinComb& lc, LabeledPoly<Engine>* lp, Randomness* lr) {
        lp->label = lc.label;
        lp->poly = eng.vzeros(0);
        for (auto& t : lc.terms) {
            auto& src = by_label.at(t.second);
            eng.vadd_scaled(lp->poly, t.first, src.first->poly);
            if (!src.second->blind.empty()) poly_add_scaled(lr->blind, t.first, src.second->blind);
        }
    };
    LabeledPoly<Engine> outer_p, inner_p;
    Randomness outer_r, inner_r;
    make_lc(outer, &outer_p, &outer_r);
    make_lc(inner, &inner_p, &inner_r);
    if (!(eng.veval(outer_p.poly, ch.beta) + outer.constant).is_zero())
        throw MarlinError("prove: outer_sumcheck linear combination does not vanish at beta");
    if (!(eng.veval(inner_p.poly, ch.gamma) + inner.constant).is_zero())
        throw MarlinError("prove: inner_sumcheck linear combination does not vanish at gamma");
    // query set, ordered by label within each point: beta {g_1, outer_sumcheck, t, z_b}; gamma {g_2, inner_sumcheck}
    std::vector<const LabeledPoly<Engine>*> at_beta = {by_label["g_1"].first, &outer_p, by_label["t"].first, by_label["z_b"].first};
    std::vector<const Randomness*> at_beta_r = {by_label["g_1"].second, &outer_r, by_label["t"].second, by_label["z_b"].second};
    std::vector<const LabeledPoly<Engine>*> at_gamma = {by_label["g_2"].first, &inner_p};
    std::vector<const Randomness*> at_gamma_r = {by_label["g_2"].second, &inner_r};
    ph.reset(); ph.reset(new ScopedPhase("r5_open"));
    proof.pc_proofs.push_back(pc_open(pk.ck, at_beta, at_beta_r, ch.beta, ch.xi));
    proof.pc_proofs.push_back(pc_open(pk.ck, at_gamma, at_gamma_r, ch.gamma, ch.xi));
    ph.reset();
    return proof;
}

// ------------------------------------------------------------------------------------------------
// verify (Marlin::verify; SURVEY 3.4) -- public input WITHOUT the leading one, padded internally
// ------------------------------------------------------------------------------------------------
// The structural checks that refuse a proof before its transcript is replayed
inline bool verify_shape(const VerifyingKey& vk, size_t n_public_inputs, const Proof& proof) {
    if (proof.commitments.size() != 3 || proof.commitments[0].size() != 4 || proof.commitments[1].size() != 3 ||
        proof.commitments[2].size() != 2 || proof.evaluations.size() != 4 || proof.pc_proofs.size() != 2)
        return false;
    if (Domain(n_public_inputs + 1).n != vk.info.num_instance || vk.index_comms.size() != 6) return false;
    return proof.commitments[1][1].has_shifted && proof.commitments[2][0].has_shifted;     // g_1 and g_2 carry degree bounds
}

// kzg10::batch_check of one proof as two flat lists of (point, scalar) terms: the proof is valid iff
//     e(sum c, h) * e(-sum w, beta_h) == 1.
// The points are the proof's own and the key's (g, gamma_g, index commitments, shift powers); the pointers stay valid
// while both live.  The opening at beta is weighted by w_beta, the one at gamma by w_gamma.
struct CheckTerms {
    std::vector<std::pair<const G1Point*, Fr>> c, w;
};
// Everything of verify up to the group arithmetic: shape checks, transcript replay, the linear combinations, the
// terms.  false when the proof is refused on the way (shape, or a degree bound without a shift power in the key).
inline bool verify_prepare(const VerifyingKey& vk, const std::vector<Fr>& public_input_unpadded, const Proof& proof,
                           const Fr& w_beta, const Fr& w_gamma, CheckTerms* out) {
    if (!verify_shape(vk, public_input_unpadded.size(), proof)) return false;
    Domain H(vk.info.num_constraints), K(vk.info.num_non_zero), X(public_input_unpadded.size() + 1);
    std::vector<Fr> public_input = public_input_unpadded;
    public_input.resize(X.n - 1, Fr::zero());
    FiatShamirRng fs;
    {
        std::vector<uint8_t> init;
        const char* name = "MARLIN-2019";
        init.insert(init.end(), name, name + 11);
        put_vk_bytes(init, vk.info, vk.index_comms);
        for (auto& x : public_input) put_fr_canonical(init, x);
        fs.initialize(init);
    }
    Challenges ch;
    fs.absorb(round_bytes(proof.commitments[0]));
    ch.alpha = sample_outside(H, fs.rng());
    ch.eta_a = rand_fr(fs.rng());
    ch.eta_b = rand_fr(fs.rng());
    ch.eta_c = rand_fr(fs.rng());
    fs.absorb(round_bytes(proof.commitments[1]));
    ch.beta = sample_outside(H, fs.rng());
    fs.absorb(round_bytes(proof.commitments[2]));
    ch.gamma = rand_fr(fs.rng());
    {
        std::vector<uint8_t> eb;
        for (auto& e : proof.evaluations) put_fr_canonical(eb, e);
        fs.absorb(eb);
    }
    uint64_t u[2];
    fs.rng().next_u128(u);
    ch.xi = fr_from_u128(u);
    LcInputs in;
    in.g1_beta = proof.evaluations[0];
    in.g2_gamma = proof.evaluations[1];
    in.t_beta = proof.evaluations[2];
    in.zb_beta = proof.evaluations[3];
    {
        std::vector<Fr> lag = X.lagrange_at(ch.beta);
        Fr acc = lag[0];                                   // the constant-one input
        for (size_t i = 1; i < X.n; i++) acc = acc + lag[i] * public_input[i - 1];
        in.x_hat_beta = acc;
        in.v_x_beta = X.vanishing_at(ch.beta);
    }
    LinComb outer, inner;
    build_lcs(H, K, ch, in, &outer, &inner);
    std::map<std::string, const Commitment*> comm;
    const char* r1[4] = {"w", "z_a", "z_b", "mask_poly"};
    const char* r2[3] = {"t", "g_1", "h_1"};
    const char* r3[2] = {"g_2", "h_2"};
    const char* ix[6] = {"row", "col", "a_val", "b_val", "c_val", "row_col"};
    for (int i = 0; i < 4; i++) comm[r1[i]] = &proof.commitments[0][i];
    for (int i = 0; i < 3; i++) comm[r2[i]] = &proof.commitments[1][i];
    for (int i = 0; i < 2; i++) comm[r3[i]] = &proof.commitments[2][i];
    for (int i = 0; i < 6; i++) comm[ix[i]] = &vk.index_comms[i];
    struct Item { const Commitment* c; const LinComb* lc; Fr value; bool bounded; size_t bound; };
    // kzg10::batch_check: total_c = sum r_i (C_i - v_i g - v'_i gamma_g + z_i W_i), total_w = sum r_i W_i,
    // r_0 = 1, r_i = u128::rand(rng); accept iff e(total_c, h) == e(total_w, beta_h).
    // Every C_i is itself a combination of commitments (accumulate_commitments_and_values with the per-polynomial
    // opening challenge powers; the two virtual commitments are linear combinations of index and prover commitments),
    // so both sums are flattened into ONE list of (point, scalar) terms each: the group elements are the ones the
    // nested scalar multiplications would give.
    std::vector<std::pair<const G1Point*, Fr>>& terms_c = out->c;
    std::vector<std::pair<const G1Point*, Fr>>& terms_w = out->w;
    terms_c.clear();
    terms_w.clear();
    bool ok = true;
    auto accumulate_point = [&](const std::vector<Item>& items, const Fr& z, const PcProof& pr, const Fr& randomizer) {
        Fr cv = Fr::zero(), chal = Fr::one();
        for (auto& it : items) {
            const Fr s = chal * randomizer;
            if (it.lc) {
                for (auto& t : it.lc->terms) terms_c.push_back({&comm.at(t.second)->comm, t.first * s});
            } else {
                terms_c.push_back({&it.c->comm, s});
            }
            cv = cv + it.value * chal;
            chal = chal * ch.xi;
            if (it.bounded) {
                // (shifted_comm - value * beta^(D - bound) g) * next challenge power
                const G1Point* sp = vk.shift_power(it.bound);
                if (!sp) { ok = false; return; }
                terms_c.push_back({&it.c->shifted, chal * randomizer});
                terms_c.push_back({sp, (it.value * chal * randomizer).neg()});
                chal = chal * ch.xi;
            }
        }
        terms_c.push_back({&vk.g, (cv * randomizer).neg()});
        if (pr.has_random_v) terms_c.push_back({&vk.gamma_g, (pr.random_v * randomizer).neg()});
        terms_c.push_back({&pr.w, z * randomizer});
        terms_w.push_back({&pr.w, randomizer});
    };
    std::vector<Item> at_beta = {{comm["g_1"], nullptr, in.g1_beta, true, H.n - 2},
                                 {nullptr, &outer, outer.constant.neg(), false, 0},
                                 {comm["t"], nullptr, in.t_beta, false, 0},
                                 {comm["z_b"], nullptr, in.zb_beta, false, 0}};
    std::vector<Item> at_gamma = {{comm["g_2"], nullptr, in.g2_gamma, true, K.n - 2}, {nullptr, &inner, inner.constant.neg(), false, 0}};
    accumulate_point(at_beta, ch.beta, proof.pc_proofs[0], w_beta);
    if (ok) accumulate_point(at_gamma, ch.gamma, proof.pc_proofs[1], w_gamma);
    return ok;
}

// The single-proof check: one u128 from rng folds the two openings (drawn once the proof has passed verify_shape), one
// host MSM per side, one pairing product
inline bool verify(const VerifyingKey& vk, const std::vector<Fr>& public_input_unpadded, const Proof& proof, ChaChaRng& rng) {
    if (!verify_shape(vk, public_input_unpadded.size(), proof)) return false;
    uint64_t rw[2];
    rng.next_u128(rw);
    CheckTerms t;
    if (!verify_prepare(vk, public_input_unpadded, proof, Fr::one(), fr_from_u128(rw), &t)) return false;
    auto values = [](const std::vector<std::pair<const G1Point*, Fr>>& in) {
        std::vector<std::pair<G1Point, Fr>> v;
        v.reserve(in.size());
        for (auto& t : in) v.push_back({*t.first, t.second});
        return v;
    };
    const G1Xyzz total_c = g1_msm_host(values(t.c)), total_w = g1_msm_host(values(t.w));
    return pairing_product_is_one({{to_affine(total_c), vk.h}, {g1_neg(to_affine(total_w)), vk.beta_h}});
}

}  // namespace marlin
}  // namespace swb
