// Host-side G1 / field helpers for the protocol layer: the parts of ark-ec / ark-ff / ark-serialize
// that Marlin's setup, transcript and (de)serialisation need outside the MSM/NTT kernels.
// Restates: short_weierstrass_jacobian::{GroupAffine::get_point_from_x, scale_by_cofactor},
// `UniformRand for GroupProjective`, Fp sqrt (Tonelli-Shanks), ToBytes (uncompressed) and
// CanonicalSerialize (compressed) for Fr / G1Affine (SURVEY A.2, A.3, row a7).
#pragma once
#include <vector>

#include "../../../include/swb200.h"
#include "../g1_decode.cuh"
#include "rng.hpp"

namespace swb {
namespace marlin {

struct G1Point {            // affine, Montgomery coordinates; GroupAffine::zero() = (0, 0, true)... kept as (0,0)
    Fq x, y;
    bool infinity = true;
    static G1Point identity() {
        G1Point p;
        p.x = Fq::zero();
        p.y = Fq::zero();
        p.infinity = true;
        return p;
    }
    bool operator==(const G1Point& o) const {
        if (infinity || o.infinity) return infinity == o.infinity;
        return x == o.x && y == o.y;
    }
};

inline G1Xyzz to_xyzz(const G1Point& p) {
    G1Xyzz r = G1Xyzz::identity();
    if (!p.infinity) {
        r.x = p.x;
        r.y = p.y;
        r.zz = Fq::one();
        r.zzz = Fq::one();
    }
    return r;
}
inline G1Point to_affine(const G1Xyzz& p) {
    G1Point r = G1Point::identity();
    if (p.is_identity()) return r;
    Fq inv = (p.zz * p.zzz).inverse_bingcd();
    r.x = p.x * (p.zzz * inv);
    r.y = p.y * (p.zz * inv);
    r.infinity = false;
    return r;
}
// an MSM result of the library: the affine value as a Z = 1 Jacobian, Z = 0 for the identity
inline G1Point from_jacobian(const swb_g1_jacobian& o) {
    G1Point p = G1Point::identity();
    Fq z;
    memcpy(z.l, o.z.l, 48);
    if (!z.is_zero()) {
        p.infinity = false;
        memcpy(p.x.l, o.x.l, 48);
        memcpy(p.y.l, o.y.l, 48);
    }
    return p;
}
inline G1Point g1_generator() {
    const uint32_t gx[12] = SWB_FQ_G1_GEN_X_INIT, gy[12] = SWB_FQ_G1_GEN_Y_INIT;
    G1Point p;
    for (int i = 0; i < 12; i++) { p.x.l[i] = gx[i]; p.y.l[i] = gy[i]; }
    p.infinity = false;
    return p;
}
inline G1Point g1_neg(const G1Point& p) {
    G1Point r = p;
    if (!p.infinity) r.y = p.y.neg();
    return r;
}
inline G1Point g1_add(const G1Point& a, const G1Point& b) {
    G1Xyzz s = to_xyzz(a);
    if (!b.infinity) s.add_affine(b.x, b.y);
    return to_affine(s);
}
// k given as little-endian 32-bit words (canonical integer)
inline G1Xyzz g1_mul_words(const G1Point& p, const uint32_t* k, int nwords) {
    G1Xyzz acc = G1Xyzz::identity();
    if (p.infinity) return acc;
    for (int i = nwords * 32 - 1; i >= 0; i--) {
        acc = acc.dbl();
        if ((k[i >> 5] >> (i & 31)) & 1u) acc.add_affine(p.x, p.y);
    }
    return acc;
}
inline G1Point g1_mul_fr(const G1Point& p, const Fr& k_mont) {
    Fr c = k_mont.to_canonical();
    return to_affine(g1_mul_words(p, c.l, 8));
}

// sum_i [k_i] P_i on the host for a handful of points (the verifier's commitments): Straus with 4-bit windows --
// one table of 15 multiples per point, the doublings shared by all of them.  36 terms: 5x fewer field products than
// 36 separate double-and-add ladders (and no inversion per term).
inline G1Xyzz g1_msm_host(const std::vector<std::pair<G1Point, Fr>>& terms) {
    std::vector<std::vector<G1Xyzz>> tab;           // tab[i][d - 1] = [d] P_i, d = 1 .. 15
    std::vector<Fr> ks;
    for (auto& t : terms) {
        if (t.first.infinity) continue;
        const Fr c = t.second.to_canonical();
        if (c.is_zero()) continue;
        std::vector<G1Xyzz> row(15);
        row[0] = to_xyzz(t.first);
        for (int d = 1; d < 15; d++) {
            row[d] = row[d - 1];
            row[d].add_affine(t.first.x, t.first.y);
        }
        tab.push_back(std::move(row));
        ks.push_back(c);
    }
    G1Xyzz acc = G1Xyzz::identity();
    for (int w = 63; w >= 0; w--) {
        if (w != 63)
            for (int k = 0; k < 4; k++) acc = acc.dbl();
        for (size_t i = 0; i < tab.size(); i++) {
            const uint32_t d = (ks[i].l[w >> 3] >> ((w & 7) * 4)) & 15u;
            if (d) acc.add(tab[i][d - 1]);
        }
    }
    return acc;
}

// ---- Fq square roots ------------------------------------------------------------------------
struct FqSqrtCtx {
    FqSqrtConsts k;         // what fq_sqrt_ts (g1_decode.cuh) needs: (t - 1) / 2 and z = 5^t, t = (q - 1) / 2^46
    FqSqrtCtx() {
        uint32_t qm1[12], t[12];
        for (int i = 0; i < 12; i++) qm1[i] = FqParams::mod(i);
        qm1[0] -= 1;
        shr(t, qm1, 46);
        shr(k.tm1h, t, 1);      // t is odd: (t - 1) / 2 = t >> 1
        k.tm1h_bits = 0;
        for (int i = 0; i < 12 * 32; i++)
            if ((k.tm1h[i >> 5] >> (i & 31)) & 1u) k.tm1h_bits = i + 1;
        Fq five = Fq::one();
        five = five + five + five + five + five;
        k.z = pow(five, t);
    }
    static void shr(uint32_t* out, const uint32_t* in, int s) {
        for (int i = 0; i < 12; i++) {
            int w = i + s / 32, b = s % 32;
            uint64_t lo = w < 12 ? in[w] : 0, hi = w + 1 < 12 ? in[w + 1] : 0;
            out[i] = (uint32_t)(((hi << 32) | lo) >> b);
        }
    }
    static Fq pow(const Fq& a, const uint32_t* e) { return fq_pow_bits(a, e, 12 * 32); }
    // Tonelli-Shanks; returns false when a is a non-residue
    bool sqrt(const Fq& a, Fq* out) const { return fq_sqrt_ts(k, a, out); }
};
inline const FqSqrtCtx& fq_sqrt_ctx() {
    static const FqSqrtCtx c;
    return c;
}

// GroupAffine::get_point_from_x(x, greatest) for y^2 = x^3 + 1
inline bool g1_point_from_x(const Fq& x, bool greatest, G1Point* out) {
    Fq y;
    if (!g1_y_from_x(fq_sqrt_ctx().k, x, greatest, &y)) return false;
    out->x = x;
    out->y = y;
    out->infinity = false;
    return true;
}
// `UniformRand for GroupProjective`: x <- Fq::rand, greatest <- bool, until on-curve; then cofactor
inline G1Point g1_rand(ChaChaRng& rng) {
    static const uint32_t cofactor[4] = {0x00000000u, 0x00000000u, 0x30000000u, 0x170b5d44u};
    for (;;) {
        Fq x = rand_fq(rng);
        bool greatest = rng.next_bool();
        G1Point p;
        if (g1_point_from_x(x, greatest, &p)) return to_affine(g1_mul_words(p, cofactor, 4));
    }
}

// ---- bytes ------------------------------------------------------------------------------------
inline void put_fr_canonical(std::vector<uint8_t>& out, const Fr& a) {     // 32 B LE
    Fr c = a.to_canonical();
    for (int i = 0; i < 8; i++)
        for (int b = 0; b < 4; b++) out.push_back((uint8_t)(c.l[i] >> (8 * b)));
}
inline void put_fq_canonical(std::vector<uint8_t>& out, const Fq& a) {     // 48 B LE
    Fq c = a.to_canonical();
    for (int i = 0; i < 12; i++)
        for (int b = 0; b < 4; b++) out.push_back((uint8_t)(c.l[i] >> (8 * b)));
}
inline void put_u64(std::vector<uint8_t>& out, uint64_t v) {
    for (int b = 0; b < 8; b++) out.push_back((uint8_t)(v >> (8 * b)));
}
// ark_ff::ToBytes for GroupAffine: x || y || infinity  (97 bytes) -- the transcript format
// (the identity is GroupAffine::zero() = (0, 1, true) in ark-ec 0.3, so its y coordinate is written as one)
inline void put_g1_uncompressed(std::vector<uint8_t>& out, const G1Point& p) {
    put_fq_canonical(out, p.infinity ? Fq::zero() : p.x);
    put_fq_canonical(out, p.infinity ? Fq::one() : p.y);
    out.push_back(p.infinity ? 1 : 0);
}
// ark_serialize::CanonicalSerialize for GroupAffine: x with SWFlags in the top bits of the last
// byte (bit 7: y is the larger of {y, -y}; bit 6: infinity) -- the proof format
inline void put_g1_compressed(std::vector<uint8_t>& out, const G1Point& p) {
    size_t at = out.size();
    if (p.infinity) {
        put_fq_canonical(out, Fq::zero());
        out[at + 47] |= 0x40;
        return;
    }
    put_fq_canonical(out, p.x);
    if (fq_canonical_gt(p.y, p.y.neg())) out[at + 47] |= 0x80;
}
inline bool get_u64(const uint8_t*& p, const uint8_t* end, uint64_t* v) {
    if (end - p < 8) return false;
    *v = 0;
    for (int b = 0; b < 8; b++) *v |= (uint64_t)p[b] << (8 * b);
    p += 8;
    return true;
}
inline bool get_fr_canonical(const uint8_t*& p, const uint8_t* end, Fr* out) {
    if (end - p < 32) return false;
    Fr c;
    for (int i = 0; i < 8; i++) c.l[i] = (uint32_t)p[4 * i] | ((uint32_t)p[4 * i + 1] << 8) | ((uint32_t)p[4 * i + 2] << 16) | ((uint32_t)p[4 * i + 3] << 24);
    for (int i = 7; i >= 0; i--) {
        if (c.l[i] != FrParams::mod(i)) {
            if (c.l[i] > FrParams::mod(i)) return false;
            break;
        }
        if (i == 0) return false;
    }
    *out = c.from_canonical();
    p += 32;
    return true;
}
// 48 little-endian bytes (flag bits already cleared) -> Fq; false when the integer is >= q (ark-serialize
// refuses non-canonical field elements)
inline bool fq_from_canonical_bytes(const uint8_t* buf, Fq* out) {
    Fq c;
    for (int i = 0; i < 12; i++) c.l[i] = (uint32_t)buf[4 * i] | ((uint32_t)buf[4 * i + 1] << 8) | ((uint32_t)buf[4 * i + 2] << 16) | ((uint32_t)buf[4 * i + 3] << 24);
    for (int i = 11; i >= 0; i--) {
        if (c.l[i] != FqParams::mod(i)) {
            if (c.l[i] > FqParams::mod(i)) return false;
            break;
        }
        if (i == 0) return false;
    }
    *out = c.from_canonical();
    return true;
}
// [r]P == O: membership in the prime-order subgroup (GroupAffine::deserialize of ark-ec 0.3 checks
// is_in_correct_subgroup_assuming_on_curve the same way)
inline bool g1_in_subgroup_plain(const G1Point& p) {
    uint32_t r[8];
    for (int i = 0; i < 8; i++) r[i] = FrParams::mod(i);
    return g1_mul_words(p, r, 8).is_identity();
}
// The same verdict from two 64-bit multiplications (g1_decode.cuh: g1_endo_holds).  beta is the cube root of unity
// for which the identity holds on the generator, found once; the self-test compares the verdicts of both tests on
// points inside and outside G1.
struct G1EndoCtx {
    Fq beta;
    G1EndoCtx() {
        uint32_t e[12];
        for (int i = 0; i < 12; i++) e[i] = FqParams::mod(i);
        e[0] -= 1;                                              // (q - 1) / 3, exactly
        uint64_t rem = 0;
        for (int i = 11; i >= 0; i--) {
            const uint64_t cur = (rem << 32) | e[i];
            e[i] = (uint32_t)(cur / 3);
            rem = cur % 3;
        }
        Fq t = Fq::one(), b = Fq::one();
        do {                                                    // t = 2, 3, ...: the first with t^((q-1)/3) != 1
            t = t + Fq::one();
            b = FqSqrtCtx::pow(t, e);
        } while (b == Fq::one());
        const G1Point g = g1_generator();
        beta = b;
        if (!g1_endo_holds(g.x, g.y, beta)) beta = b * b;
    }
};
// the decoder's constants, computed once; the batch verifier passes the same values to its kernel
inline const G1DecodeConsts& g1_decode_consts() {
    static const G1DecodeConsts k = [] {
        G1DecodeConsts r;
        r.sq = fq_sqrt_ctx().k;
        r.beta = G1EndoCtx().beta;
        return r;
    }();
    return k;
}
inline bool g1_in_subgroup(const G1Point& p) {
    if (p.infinity) return true;
    return g1_endo_holds(p.x, p.y, g1_decode_consts().beta);
}
// CanonicalDeserialize for GroupAffine (g1_decode.cuh); p advances by 48 bytes whatever the verdict
inline bool get_g1_compressed(const uint8_t*& p, const uint8_t* end, G1Point* out) {
    if (end - p < 48) return false;
    uint32_t w[12];
    for (int i = 0; i < 12; i++)
        w[i] = (uint32_t)p[4 * i] | ((uint32_t)p[4 * i + 1] << 8) | ((uint32_t)p[4 * i + 2] << 16) | ((uint32_t)p[4 * i + 3] << 24);
    p += 48;
    Fq x, y;
    if (g1_decode(g1_decode_consts(), w, &x, &y) != G1D_OK) return false;
    out->x = x;
    out->y = y;
    out->infinity = x.is_zero() && y.is_zero();
    return true;
}

}  // namespace marlin
}  // namespace swb
