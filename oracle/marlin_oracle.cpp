/* TEST INFRASTRUCTURE ONLY -- CPU arm of the Marlin protocol, for parity and the CPU baseline.
 *
 * Instantiates the protocol templates of simpleworks_b200/csrc/marlin/ (shared source: transcript,
 * AHP rounds, KZG bookkeeping) with a CPU engine built on the C restatement of arkworks'
 * operators in oracle.c (orc_ntt, orc_msm_variable_base, orc_fixed_base_powers).  What this arm
 * pins: the CUDA engine (NTT / MSM / fixed-base kernels) yields byte-identical proofs to the CPU
 * operators under the same RNG streams.  The protocol logic itself is shared and therefore checked
 * by completeness / tamper tests, not by this arm.  PARITY UNPINNED against real arkworks.
 * The product library never links this file.
 */
#include <omp.h>

#include "marlin/c_api_impl.hpp"
#include "marlin/vec_host.hpp"
#include "swb_oracle.h"

using namespace swb;
using namespace swb::marlin;

namespace {

// multi-process proving on the CPU arm, mirroring swb_set_msm_shard: each process computes its
// contiguous share of every prover MSM and `combine` returns the sum over all processes
struct OrcShard {
    int rank = 0, world = 1;
    int (*combine)(void*, const g1_jac_t*, g1_jac_t*) = nullptr;
    void* user = nullptr;
} g_shard;

struct CpuBases {
    std::vector<g1_affine_t> pts;
};

struct CpuEngine : HostVecOps {
    void vntt(Vec& v, uint32_t log_n, bool inverse, bool coset) {
        if (v.size() != ((size_t)1 << log_n)) throw MarlinError("vntt: size mismatch");
        orc_ntt(reinterpret_cast<fr_t*>(v.data()), log_n, inverse, coset, 0);
    }
    void* bases_from_powers(const G1Point& g, const Fr& beta, size_t n) {
        auto* b = new CpuBases();
        b->pts.resize(n);
        g1_jac_t gj;
        memset(&gj, 0, sizeof gj);
        if (g.infinity) orc_g1_jac_zero(&gj);
        else {
            memcpy(gj.x.l, g.x.l, 48);
            memcpy(gj.y.l, g.y.l, 48);
            Fq one = Fq::one();
            memcpy(gj.z.l, one.l, 48);
        }
        fr_t bt;
        memcpy(bt.l, beta.l, 32);
        orc_fixed_base_powers(b->pts.data(), &gj, &bt, n, 0);
        return b;
    }
    void export_bases(void* h, size_t offset, size_t n, G1Point* out) {
        auto* b = static_cast<CpuBases*>(h);
        for (size_t i = 0; i < n; i++) {
            const g1_affine_t& a = b->pts[offset + i];
            out[i].infinity = a.infinity != 0;
            memcpy(out[i].x.l, a.x.l, 48);
            memcpy(out[i].y.l, a.y.l, 48);
        }
    }
    void free_bases(void* h) { delete static_cast<CpuBases*>(h); }
    void bases_tune(void*, size_t) {}     // nothing to restructure on the CPU arm
    size_t msm_submit(void* h, size_t offset, const Vec& scalars, size_t n) { return msm_submit_sync(*this, h, offset, scalars, n); }
    size_t msm_local_count(size_t n) {
        if (!(g_shard.world > 1 && g_shard.combine)) return n;
        return n / (size_t)g_shard.world + ((size_t)g_shard.rank < n % (size_t)g_shard.world ? 1 : 0);
    }
    G1Point msm(void* h, size_t offset_full, const Vec& scalars, size_t n_full) {
        // this process's share of the index range (all of it unless orc_set_msm_shard is active)
        const bool sharded = g_shard.world > 1 && g_shard.combine;
        size_t lo = 0, n = n_full;
        if (sharded) {
            const size_t base = n_full / (size_t)g_shard.world, rem = n_full % (size_t)g_shard.world, r = (size_t)g_shard.rank;
            lo = r * base + (r < rem ? r : rem);
            n = base + (r < rem ? 1 : 0);
        }
        const size_t offset = offset_full + lo;
        const Fr* scalars_mont = scalars.data() + lo;
        auto* b = static_cast<CpuBases*>(h);
        std::vector<big256_t> sc(n);
#pragma omp parallel for schedule(static)
        for (size_t i = 0; i < n; i++) orc_fr_to_canon(&sc[i], reinterpret_cast<const fr_t*>(&scalars_mont[i]));
        g1_jac_t out;
        orc_msm_variable_base(&out, b->pts.data() + offset, sc.data(), n, 0);
        if (sharded) {
            g1_jac_t sum;
            if (g_shard.combine(g_shard.user, &out, &sum) != 0) throw MarlinError("msm: combining the processes' partial results failed");
            out = sum;
        }
        g1_affine_t a;
        orc_g1_to_affine(&a, &out);
        G1Point p = G1Point::identity();
        if (!a.infinity) {
            p.infinity = false;
            memcpy(p.x.l, a.x.l, 48);
            memcpy(p.y.l, a.y.l, 48);
        }
        return p;
    }
};

CpuEngine g_engine;
thread_local std::string g_err;
using Api = MarlinApi<CpuEngine>;

}  // namespace

extern "C" {

const char* orc_marlin_last_error() { return g_err.c_str(); }

void* orc_rng_test_rng() {
    auto* h = new RngHandle();
    h->rng = test_rng();
    return h;
}
void* orc_rng_from_seed(const uint8_t seed[32], int rounds) {
    auto* h = new RngHandle();
    h->rng = ChaChaRng(seed, rounds);
    return h;
}
uint64_t orc_rng_next_u64(void* h) { return static_cast<RngHandle*>(h)->rng.next_u64(); }
uint32_t orc_rng_next_u32(void* h) { return static_cast<RngHandle*>(h)->rng.next_u32(); }
void orc_rng_fr_rand(void* h, uint64_t out[4]) {
    Fr r = rand_fr(static_cast<RngHandle*>(h)->rng);
    memcpy(out, r.l, 32);
}
void orc_rng_free(void* h) { delete static_cast<RngHandle*>(h); }
void orc_blake2s(const uint8_t* in, size_t n, uint8_t out[32]) {
    Blake2s s;
    s.update(in, n);
    s.finalize(out);
}

void* orc_r1cs_new(size_t ni, size_t nw) { return r1cs_new(ni, nw); }
void* orc_r1cs_builtin(int kind, size_t size, uint64_t v0, uint64_t v1) { return r1cs_builtin(kind, size, v0, v1); }
int orc_r1cs_add_constraint(void* h, const uint64_t* ac, const uint32_t* ai, size_t na, const uint64_t* bc, const uint32_t* bi,
                            size_t nb, const uint64_t* cc, const uint32_t* ci, size_t nc) {
    return r1cs_add_constraint(static_cast<R1csHandle*>(h), ac, ai, na, bc, bi, nb, cc, ci, nc);
}
int orc_r1cs_set_assignment(void* h, const uint64_t* inst, size_t ni, const uint64_t* wit, size_t nw) {
    return r1cs_set_assignment(static_cast<R1csHandle*>(h), inst, ni, wit, nw);
}
int orc_r1cs_is_satisfied(void* h) { return static_cast<R1csHandle*>(h)->cs.is_satisfied() ? 1 : 0; }
void orc_r1cs_free(void* h) { delete static_cast<R1csHandle*>(h); }

int orc_marlin_universal_setup(size_t nc, size_t nv, size_t nnz, void* rng, void** srs) {
    SrsHandle<CpuEngine>* out = nullptr;
    int rc = Api::setup(g_engine, nc, nv, nnz, static_cast<RngHandle*>(rng), &out, &g_err);
    *srs = out;
    return rc;
}
size_t orc_srs_max_degree(void* srs) { return static_cast<SrsHandle<CpuEngine>*>(srs)->srs->max_degree; }
void orc_srs_free(void* srs) { delete static_cast<SrsHandle<CpuEngine>*>(srs); }
int orc_marlin_index(void* srs, void* cs, void** pk, void** vk) {
    PkHandle<CpuEngine>* p = nullptr;
    VkHandle* v = nullptr;
    int rc = Api::index(static_cast<SrsHandle<CpuEngine>*>(srs), static_cast<R1csHandle*>(cs), &p, &v, &g_err);
    *pk = p;
    *vk = v;
    return rc;
}
void orc_pk_free(void* pk) { delete static_cast<PkHandle<CpuEngine>*>(pk); }
void orc_vk_free(void* vk) { delete static_cast<VkHandle*>(vk); }
int orc_set_msm_shard(int rank, int world, int (*combine)(void*, const g1_jac_t*, g1_jac_t*), void* user) {
    g_shard.rank = world > 1 ? rank : 0;
    g_shard.world = world > 1 && combine ? world : 1;
    g_shard.combine = world > 1 ? combine : nullptr;
    g_shard.user = user;
    return 0;
}
int orc_marlin_prove(void* pk, void* cs, void* rng, uint8_t** bytes, size_t* len) {
    return Api::prove(static_cast<PkHandle<CpuEngine>*>(pk), static_cast<R1csHandle*>(cs), static_cast<RngHandle*>(rng), bytes, len,
                      &g_err);
}
int orc_marlin_verify(void* vk, const uint64_t* pi, size_t n, const uint8_t* proof, size_t len, void* rng, int* ok) {
    return Api::verify(static_cast<VkHandle*>(vk), pi, n, proof, len, static_cast<RngHandle*>(rng), ok, &g_err);
}
void orc_bytes_free(uint8_t* p) { free(p); }
void* orc_r1cs_read(const uint8_t* b, size_t n) { return r1cs_from_bytes(b, n); }
uint8_t* orc_r1cs_write(void* h, size_t* len) { return r1cs_to_bytes(static_cast<R1csHandle*>(h), len); }
uint8_t* orc_vk_serialize(void* vk, size_t* len) { return vk_to_bytes(static_cast<VkHandle*>(vk), len); }
void* orc_vk_deserialize(const uint8_t* b, size_t n) { return vk_from_bytes(b, n); }

/* self-test of the pairing tower used by the verifier: field inverses, tower relations, a G2 point
 * of order r from the derived cofactor, bilinearity, non-degeneracy, the product check; returns a
 * bit mask of failed checks */
int orc_pairing_selftest() {
    ChaChaRng rng = test_rng();
    int bad = 0;
    Fq2 a2 = {rand_fq(rng), rand_fq(rng)};
    if (!(a2 * a2.inverse() == Fq2::one())) bad |= 1;
    Fq6 a6 = {{rand_fq(rng), rand_fq(rng)}, {rand_fq(rng), rand_fq(rng)}, {rand_fq(rng), rand_fq(rng)}};
    if (!(a6 * a6.inverse() == Fq6::one())) bad |= 2;
    Fq12 a12 = {a6, a6 * a6};
    if (!(a12 * a12.inverse() == Fq12::one())) bad |= 4;
    Fq6 v = Fq6::zero();
    v.c1 = Fq2::one();
    Fq6 uu = Fq6::zero();
    uu.c0 = {Fq::zero(), Fq::one()};
    if (!(v * v * v == uu)) bad |= 8;
    Fq2 sq = a2.sqr(), r;
    if (!fq2_sqrt(sq, &r) || !(r.sqr() == sq)) bad |= 16;
    G2Point h = g2_rand(rng);
    uint32_t rw[8];
    for (int i = 0; i < 8; i++) rw[i] = FrParams::mod(i);
    if (!g2_on_curve(h) || h.infinity || !g2_mul_words(h, rw, 8).infinity) bad |= 32;
    G1Point g = g1_generator();
    Fr a = rand_fr(rng), b = rand_fr(rng);
    Fq12 e = pairing(g, h);
    if (e == Fq12::one()) bad |= 64;
    Fr ab = (a * b).to_canonical();
    if (!(pairing(g1_mul_fr(g, a), g2_mul_fr(h, b)) == e.pow_words(ab.l, 8))) bad |= 128;
    if (!(e.pow_words(rw, 8) == Fq12::one())) bad |= 256;
    if (!pairing_product_is_one({{g1_mul_fr(g, a), h}, {g1_neg(g), g2_mul_fr(h, a)}})) bad |= 512;
    if (pairing_product_is_one({{g1_mul_fr(g, a), h}, {g1_neg(g), g2_mul_fr(h, b)}})) bad |= 1024;
    // Frobenius is the q-th power; the fast final exponentiation is the cube of the plain one
    uint32_t qw[12];
    for (int i = 0; i < 12; i++) qw[i] = FqParams::mod(i);
    if (!(frobenius(a12) == a12.pow_words(qw, 12))) bad |= 2048;
    if (!(frobenius(a12, 2) == a12.pow_words(qw, 12).pow_words(qw, 12))) bad |= 4096;
    const Fq12 ml = miller_loop(g1_mul_fr(g, a), h);
    const Fq12 plain = final_exponentiation_plain(ml);
    if (!(final_exponentiation(ml) == plain * plain * plain)) bad |= 8192;
    const Fq12 plain2 = final_exponentiation_plain(a12);
    if (!(final_exponentiation(a12) == plain2 * plain2 * plain2)) bad |= 16384;
    // the Miller loop on the twist (Fq2 steps, sparse lines) gives the values of the loop over E(Fq12), bit for bit
    for (int k = 0; k < 3; k++) {
        const G1Point pk = g1_mul_fr(g, rand_fr(rng));
        const G2Point qk = g2_mul_fr(h, rand_fr(rng));
        const Fq12 plain_k = miller_loop_plain(pk, qk);
        if (!(miller_loop_affine(pk, qk) == plain_k)) bad |= 32768;
        // the projective loop scales its lines by Fq2 factors: equal after the final exponentiation
        if (!(final_exponentiation(miller_loop(pk, qk)) == final_exponentiation(plain_k))) bad |= 65536;
        const Fq12 sq = plain_k.sqr();
        if (!(sq == plain_k * plain_k)) bad |= 131072;
    }
    // the projective G2 ladder gives the affine ladder's points (cofactor-sized and field-sized scalars, small ones, zero)
    {
        static const uint32_t cof[SWB_G2_COFACTOR_WORDS] = SWB_G2_COFACTOR_INIT;
        if (!(g2_mul_words(h, cof, SWB_G2_COFACTOR_WORDS) == g2_mul_words_affine(h, cof, SWB_G2_COFACTOR_WORDS))) bad |= 2097152;
        for (uint32_t kk = 0; kk < 6; kk++) {
            uint32_t w[8] = {kk, 0, 0, 0, 0, 0, 0, 0};
            if (kk == 5) for (int i = 0; i < 8; i++) w[i] = rw[i] - (i == 0 ? 1u : 0u);          // r - 1: -Q
            if (!(g2_mul_words(h, w, 8) == g2_mul_words_affine(h, w, 8))) bad |= 2097152;
        }
        const Fr kf = rand_fr(rng).to_canonical();
        if (!(g2_mul_words(h, kf.l, 8) == g2_mul_words_affine(h, kf.l, 8))) bad |= 2097152;
    }
    // cyclotomic squaring equals the plain one on the cyclotomic subgroup (elements after the easy part)
    {
        Fq12 c = a12.conj() * a12.inverse();
        c = frobenius(c, 2) * c;
        for (int k = 0; k < 4; k++) {
            if (!(c.cyclotomic_sqr() == c.sqr())) bad |= 16777216;
            c = c * c.sqr();
        }
        if (!(exp_by_x(c, true) == exp_by_x(c, false))) bad |= 16777216;
    }
    // the shared-squaring loop over several pairs is the product of the single loops
    {
        const G1Point p1 = g1_mul_fr(g, rand_fr(rng)), p2 = g1_mul_fr(g, rand_fr(rng));
        const G2Point q1 = g2_mul_fr(h, rand_fr(rng)), q2 = g2_mul_fr(h, rand_fr(rng));
        if (!(miller_loop_multi({{p1, q1}, {p2, q2}, {G1Point::identity(), q1}}) == miller_loop(p1, q1) * miller_loop(p2, q2))) bad |= 8388608;
        if (!(miller_loop_multi({}) == Fq12::one())) bad |= 8388608;
    }
    // the verifier's host MSM (Straus, shared doublings) equals the sum of separate scalar multiplications, with
    // zero scalars, the identity, repeated and negated points among the terms
    {
        std::vector<std::pair<G1Point, Fr>> terms;
        G1Xyzz want = G1Xyzz::identity();
        for (int k = 0; k < 9; k++) {
            G1Point pt = k == 3 ? G1Point::identity() : g1_mul_fr(g, rand_fr(rng));
            if (k == 5) pt = terms[1].first;
            if (k == 6) pt = g1_neg(terms[1].first);
            Fr sc = k == 2 ? Fr::zero() : rand_fr(rng);
            if (k == 6) sc = terms[5].second;                      // cancels term 5
            if (k == 7) sc = Fr::one();
            if (k == 8) sc = Fr::zero() - Fr::one();               // r - 1
            terms.push_back({pt, sc});
            const G1Point part = g1_mul_fr(pt, sc);
            if (!part.infinity) want.add_affine(part.x, part.y);
        }
        if (!(to_affine(g1_msm_host(terms)) == to_affine(want))) bad |= 4194304;
        if (!g1_msm_host({}).is_identity()) bad |= 4194304;
    }
    // subgroup membership by the endomorphism agrees with [r]P == O: on multiples of the generator, on random curve
    // points (outside G1 with overwhelming probability: the cofactor has 125 bits) and on their cofactor-cleared images
    {
        int inside = 0, outside = 0;
        for (int k = 0; k < 12; k++) {
            G1Point c;
            Fq xk = rand_fq(rng);
            if (!g1_point_from_x(xk, (k & 1) != 0, &c)) continue;
            const bool a1 = g1_in_subgroup(c), a2 = g1_in_subgroup_plain(c);
            if (a1 != a2) bad |= 262144;
            (a2 ? inside : outside)++;
            const G1Point m = g1_mul_fr(g, rand_fr(rng));
            if (!g1_in_subgroup(m) || !g1_in_subgroup_plain(m)) bad |= 524288;
        }
        if (outside == 0) bad |= 1048576;                      // the test must have seen points outside G1
    }
    return bad;
}

}  // extern "C"
