// Decompression of ark-serialize compressed G1 points (48 bytes: x little-endian, SWFlags in the top two bits of the
// last byte -- bit 7: y is the larger of {y, -y}, bit 6: the identity), with the subgroup test that
// GroupAffine::deserialize applies.  One piece of code for the host parser (marlin/curve_host.hpp: get_g1_compressed)
// and the batch verifier's kernel (verify_ops.cu), so both give the same verdict on every input.  Nothing decoded here
// is secret: the loops run in variable time.
#pragma once
#include "g1.cuh"

namespace swb {

// Tonelli-Shanks constants of Fq (q - 1 = 2^46 t, t odd), computed once on the host (marlin/curve_host.hpp)
struct FqSqrtConsts {
    uint32_t tm1h[12];      // (t - 1) / 2
    int tm1h_bits;          // its bit length
    Fq z;                   // 5^t: generator of the 2-Sylow subgroup (5 is a non-residue)
};
// everything the decoder needs besides the encoding
struct G1DecodeConsts {
    FqSqrtConsts sq;
    Fq beta;                // the cube root of unity with phi(P) = (beta x, y) = -[x^2]P on G1 (x: the BLS parameter)
};

// verdicts of g1_decode; G1D_OK for every point get_g1_compressed accepts, the identity included
enum G1DecodeStatus : uint8_t {
    G1D_OK = 0,
    G1D_BAD_IDENTITY = 1,   // infinity flag with a sign bit or a non-zero x: the identity has one encoding
    G1D_NOT_REDUCED = 2,    // x >= q
    G1D_NOT_ON_CURVE = 3,   // x^3 + 1 is not a square
    G1D_NOT_IN_G1 = 4,      // on the curve, outside the prime-order subgroup
};

// a^e, e given as little-endian words of `bits` significant bits
SWB_HD Fq fq_pow_bits(const Fq& a, const uint32_t* e, int bits) {
    Fq acc = Fq::one();
    for (int i = bits - 1; i >= 0; i--) {
        acc = acc.sqr();
        if ((e[i >> 5] >> (i & 31)) & 1u) acc = acc * a;
    }
    return acc;
}

// A square root of a (Tonelli-Shanks); false when a is a non-residue.  One exponentiation w = a^((t-1)/2) gives both
// starting values, x = a w = a^((t+1)/2) and b = x w = a^t.  For a residue b^(2^45) = a^((q-1)/2) = 1, so b has order at
// most 2^45 and every round of the loop finds the order of b below 2^m; a non-residue's b has order exactly 2^46, which
// the first round detects -- no separate Legendre symbol.
SWB_HD bool fq_sqrt_ts(const FqSqrtConsts& k, const Fq& a, Fq* out) {
    if (a.is_zero()) { *out = a; return true; }
    const Fq one = Fq::one();
    const Fq w = fq_pow_bits(a, k.tm1h, k.tm1h_bits);
    Fq x = a * w;
    Fq b = x * w;
    Fq zz = k.z;
    int m = 46;
    while (!(b == one)) {
        int i = 0;
        Fq b2 = b;
        while (!(b2 == one)) {
            if (i == m - 1) return false;
            b2 = b2.sqr();
            i++;
        }
        Fq t = zz;
        for (int j = 0; j < m - i - 1; j++) t = t.sqr();
        zz = t.sqr();
        b = b * zz;
        x = x * t;
        m = i;
    }
    *out = x;
    return true;
}

// canonical integer comparison a > b (both Montgomery)
SWB_HD bool fq_canonical_gt(const Fq& a, const Fq& b) {
    const Fq ca = a.to_canonical(), cb = b.to_canonical();
    for (int i = 11; i >= 0; i--)
        if (ca.l[i] != cb.l[i]) return ca.l[i] > cb.l[i];
    return false;
}

// GroupAffine::get_point_from_x(x, greatest) for y^2 = x^3 + 1: the y of the requested sign, false when x is not the
// abscissa of a curve point
SWB_HD bool g1_y_from_x(const FqSqrtConsts& k, const Fq& x, bool greatest, Fq* y) {
    const Fq rhs = x.sqr() * x + Fq::one();
    Fq r;
    if (!fq_sqrt_ts(k, rhs, &r)) return false;
    const Fq negr = r.neg();
    const bool r_lt_negr = fq_canonical_gt(negr, r);
    *y = (r_lt_negr ^ greatest) ? r : negr;
    return true;
}

// [k]P for an affine point P and a 64-bit k (double-and-add from the top bit)
SWB_HD G1Xyzz g1_mul_u64(const Fq& px, const Fq& py, uint64_t k) {
    G1Xyzz acc = G1Xyzz::identity();
    for (int i = 63; i >= 0; i--) {
        acc = acc.dbl();
        if ((k >> i) & 1u) acc.add_affine(px, py);
    }
    return acc;
}

// Membership of the curve point (px, py) != O in G1 (Scott, "A note on group membership tests for G1, G2 and GT on BLS
// pairing-friendly curves"; what ark-bls12-377 0.4 does): P is in G1 iff phi(P) = -[x^2]P, where phi(X, Y) = (beta X, Y)
// is the curve's order-3 endomorphism and x the BLS parameter
SWB_HD bool g1_endo_holds(const Fq& px, const Fq& py, const Fq& beta) {
    const G1Xyzz xp = g1_mul_u64(px, py, SWB_BLS_X);
    if (xp.is_identity()) return false;
    const Fq inv = (xp.zz * xp.zzz).inverse_bingcd();
    const Fq ax = xp.x * (xp.zzz * inv), ay = xp.y * (xp.zz * inv);
    if (ax == px && ay == py) return false;                    // [x]P = P: not of order r
    const G1Xyzz x2 = g1_mul_u64(ax, ay, SWB_BLS_X);           // [x^2]P must be (beta X, -Y)
    if (x2.is_identity()) return false;
    return x2.x == (beta * px) * x2.zz && x2.y == py.neg() * x2.zzz;
}

// One compressed encoding, as 12 little-endian words, to the swb_bases record (x, y) in Montgomery form: the identity
// as (0, 0), which no curve point has; (0, 0) also for every refused encoding
SWB_HD uint8_t g1_decode(const G1DecodeConsts& k, const uint32_t* enc, Fq* ox, Fq* oy) {
    *ox = Fq::zero();
    *oy = Fq::zero();
    Fq c;
    for (int i = 0; i < 12; i++) c.l[i] = enc[i];
    const uint32_t flags = enc[11] >> 30;
    c.l[11] &= 0x3FFFFFFFu;
    if (flags & 1u) {
        // the identity has one encoding: x = 0, no sign bit (stricter than upstream, which ignores x here)
        return (flags & 2u) || !c.is_zero() ? G1D_BAD_IDENTITY : G1D_OK;
    }
    for (int i = 11; i >= 0; i--) {                            // ark-serialize refuses x >= q
        if (c.l[i] != FqParams::mod(i)) {
            if (c.l[i] > FqParams::mod(i)) return G1D_NOT_REDUCED;
            break;
        }
        if (i == 0) return G1D_NOT_REDUCED;
    }
    const Fq x = c.from_canonical();
    Fq y;
    if (!g1_y_from_x(k.sq, x, (flags & 2u) != 0, &y)) return G1D_NOT_ON_CURVE;
    if (!g1_endo_holds(x, y, k.beta)) return G1D_NOT_IN_G1;
    *ox = x;
    *oy = y;
    return G1D_OK;
}

}  // namespace swb
