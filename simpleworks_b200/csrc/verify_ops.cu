// Batch verification of Marlin proofs (swb_marlin_verify_batch).
//
// Every proof's check is e(A_j, h) * e(-B_j, beta_h) = 1, A_j and B_j the G1 sums of marlin::verify_prepare.  Proofs whose
// keys share (h, beta_h) -- every key indexed from one SRS -- fold into one such equation with independent secret 128-bit
// weights rho_j: e(sum rho_j A_j, h) * e(-sum rho_j B_j, beta_h) = 1.  So a batch costs two Miller loops per pairing group
// and one final exponentiation; per proof there remain the decoding of its G1 points (a square root and a subgroup test
// each: k_g1_decode, one thread per point), the transcript replay (host, in parallel) and its share of two MSMs over
// all proof points (the library's MSM pipeline).  When the equation fails, halves of the undecided proofs are checked
// the same way until every invalid proof stands alone: O(f log n) sub-checks for f invalid proofs.  For any fixed set
// holding a wrong proof, its equation holds with probability about 2^-127 over the weights, so the sub-checks reuse them.
#include <algorithm>
#include <functional>
#include <numeric>

#include "verify_ops.hpp"

namespace swb {

__global__ void __launch_bounds__(128) k_g1_decode(const uint32_t* __restrict__ enc, size_t n, const G1DecodeConsts k,
                                                   Fq* __restrict__ xy, uint8_t* __restrict__ status) {
    const size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t w[12];
#pragma unroll
    for (int j = 0; j < 12; j++) w[j] = enc[12 * i + j];
    Fq x, y;
    status[i] = g1_decode(k, w, &x, &y);
    xy[2 * i] = x;
    xy[2 * i + 1] = y;
}

int g1_decode_dev(swb_ctx* c, const uint32_t* enc_dev, size_t n, const G1DecodeConsts& k, Fq* xy_dev, uint8_t* status_dev) {
    if (n == 0) return SWB_OK;
    SWB_REQUIRE(c, enc_dev && xy_dev && status_dev, "g1_decode: NULL buffer");
    SWB_CUDA(c, cudaSetDevice(c->device));
    k_g1_decode<<<(unsigned)((n + 127) / 128), 128, 0, c->stream>>>(enc_dev, n, k, xy_dev, status_dev);
    SWB_LAUNCH_CHECK(c, "k_g1_decode");
    return SWB_OK;
}

namespace {

using namespace marlin;
using Terms = std::vector<std::pair<const G1Point*, Fr>>;

struct BatchProof {
    Proof pr;
    std::vector<G1Point*> pts;              // the proof's points in encoding order: what the decoder fills in
    std::vector<const uint8_t*> enc;        // their encodings
    bool live = false;                      // parsed, decoded and prepared: undecided until a pairing check
    Terms key_terms;                        // scalars of the key's points, summed per point
};

// the index of p among pts, or -1 (a point of the key)
long position_of(const std::vector<G1Point*>& pts, const G1Point* p) {
    for (size_t i = 0; i < pts.size(); i++)
        if (pts[i] == p) return (long)i;
    return -1;
}
void add_term(Terms& ts, const G1Point* p, const Fr& s) {
    for (auto& t : ts)
        if (t.first == p) { t.second = t.second + s; return; }
    ts.push_back({p, s});
}
// runs body(j) for j < n on all cores; the first exception is rethrown afterwards
template <class F>
void parallel_for(size_t n, F&& body) {
    std::string err;
    bool failed = false;
#pragma omp parallel for schedule(dynamic, 8)
    for (long j = 0; j < (long)n; j++) {
        try {
            body((size_t)j);
        } catch (const std::exception& e) {
#pragma omp critical(swb_verify_batch_err)
            if (!failed) { failed = true; err = e.what(); }
        }
    }
    if (failed) throw MarlinError(err);
}

}  // namespace

int marlin_verify_batch(swb_ctx* c, size_t n, const VerifyingKey* const* vks, const uint64_t* const* public_inputs, const size_t* n_inputs,
                        const uint8_t* const* proofs, const size_t* lens, ChaChaRng& rng, int* ok) {
    SWB_CUDA(c, cudaSetDevice(c->device));
    StageTimer st(c, "verify_batch");
    std::vector<Fr> rho(n), fold(n);
    for (size_t j = 0; j < n; j++) {
        uint64_t u[2];
        rng.next_u128(u);
        rho[j] = fr_from_u128(u);
        rng.next_u128(u);
        fold[j] = rho[j] * fr_from_u128(u);       // weight of the proof's opening at gamma
    }
    // pairing groups: keys with the same (h, beta_h).  The proofs are laid out group by group (`order`), so that the points
    // of any run of proofs inside one group form one contiguous range of the bases.
    std::vector<const VerifyingKey*> group_key;
    std::vector<size_t> group(n);
    for (size_t j = 0; j < n; j++) {
        size_t g = 0;
        while (g < group_key.size() && !(group_key[g] == vks[j] || (group_key[g]->h == vks[j]->h && group_key[g]->beta_h == vks[j]->beta_h))) g++;
        if (g == group_key.size()) group_key.push_back(vks[j]);
        group[j] = g;
    }
    std::vector<size_t> order(n);
    std::iota(order.begin(), order.end(), (size_t)0);
    std::stable_sort(order.begin(), order.end(), [&](size_t a, size_t b) { return group[a] < group[b]; });

    // ---- parse: the proof layout and its field elements on the host, the point encodings collected ----------------
    std::vector<BatchProof> bp(n);
    parallel_for(n, [&](size_t j) {
        BatchProof& b = bp[j];
        auto collect = [&b](const uint8_t*& p, const uint8_t* end, G1Point* out) {
            if (end - p < 48) return false;
            b.pts.push_back(out);
            b.enc.push_back(p);
            p += 48;
            return true;
        };
        b.live = Proof::deserialize(proofs[j], lens[j], &b.pr, collect);
        if (!b.live) {
            b.pts.clear();
            b.enc.clear();
        }
    });
    std::vector<size_t> base(n + 1);                 // base[k]: first point of the proof at layout position k
    base[0] = 0;
    for (size_t k = 0; k < n; k++) base[k + 1] = base[k] + bp[order[k]].pts.size();
    const size_t total = base[n];
    st.mark("parse");

    // ---- decode: all points in one launch; back to the host, since the transcripts absorb uncompressed points --------
    uint32_t* enc_dev = static_cast<uint32_t*>(get_scratch(c, "verify_enc", total * 48 + 64));
    Fq* xy_dev = static_cast<Fq*>(get_scratch(c, "verify_xy", total * 96 + 64));
    uint8_t* status_dev = static_cast<uint8_t*>(get_scratch(c, "verify_status", total + 64));
    if (!enc_dev || !xy_dev || !status_dev) return SWB_ENOMEM;
    std::vector<uint32_t> enc(total * 12);
    std::vector<Fq> xy(total * 2);
    std::vector<uint8_t> status(total);
    parallel_for(n, [&](size_t k) {
        const BatchProof& b = bp[order[k]];
        for (size_t i = 0; i < b.enc.size(); i++) memcpy(&enc[(base[k] + i) * 12], b.enc[i], 48);
    });
    if (total) {
        SWB_CUDA(c, cudaMemcpyAsync(enc_dev, enc.data(), total * 48, cudaMemcpyHostToDevice, c->stream));
        int rc = g1_decode_dev(c, enc_dev, total, g1_decode_consts(), xy_dev, status_dev);
        if (rc != SWB_OK) return rc;
        SWB_CUDA(c, cudaMemcpyAsync(xy.data(), xy_dev, total * 96, cudaMemcpyDeviceToHost, c->stream));
        SWB_CUDA(c, cudaMemcpyAsync(status.data(), status_dev, total, cudaMemcpyDeviceToHost, c->stream));
        SWB_CUDA(c, cudaStreamSynchronize(c->stream));
    }
    st.mark("decode");

    // ---- transcripts: the points into the proofs, verify_prepare, the scalars of every term ---------------------------
    std::vector<Fr> sc(2 * total, Fr::zero());       // [0, total): sum A; [total, 2 total): sum B -- per point
    parallel_for(n, [&](size_t k) {
        const size_t j = order[k];
        BatchProof& b = bp[j];
        for (size_t i = 0; b.live && i < b.pts.size(); i++) {
            const size_t at = base[k] + i;
            if (status[at] != G1D_OK) { b.live = false; break; }
            G1Point& p = *b.pts[i];
            p.x = xy[2 * at];
            p.y = xy[2 * at + 1];
            p.infinity = p.x.is_zero() && p.y.is_zero();
        }
        if (!b.live) return;
        std::vector<Fr> pi(n_inputs[j]);
        for (size_t i = 0; i < pi.size(); i++) memcpy(pi[i].l, public_inputs[j] + 4 * i, sizeof(Fr));
        CheckTerms t;
        if (!verify_prepare(*vks[j], pi, b.pr, rho[j], fold[j], &t)) { b.live = false; return; }
        for (int side = 0; side < 2; side++) {
            for (auto& term : side ? t.w : t.c) {
                const long s = position_of(b.pts, term.first);
                if (s < 0) add_term(b.key_terms, term.first, term.second);      // only A has key points
                else if (!term.first->infinity) {
                    Fr& dst = sc[side * total + base[k] + (size_t)s];
                    dst = dst + term.second;
                }
            }
        }
    });
    std::vector<size_t> live_before(n + 1, 0);      // live proofs at layout positions < k
    for (size_t k = 0; k < n; k++) live_before[k + 1] = live_before[k] + (bp[order[k]].live ? 1 : 0);
    Fr* sc_dev = static_cast<Fr*>(get_scratch(c, "verify_scalars", 2 * total * sizeof(Fr) + 64));
    if (!sc_dev) return SWB_ENOMEM;
    if (total) SWB_CUDA(c, cudaMemcpyAsync(sc_dev, sc.data(), 2 * total * sizeof(Fr), cudaMemcpyHostToDevice, c->stream));
    st.mark("transcripts");

    // ---- the folded check of the live proofs at layout positions [lo, hi) --------------------------------------------
    swb_bases bases;                                 // the decoded points, device-resident, contiguous per proof
    bases.ctx = c;
    bases.xy = xy_dev;
    bases.n = total;
    std::vector<size_t> group_start(group_key.size() + 1, n);
    for (size_t k = n; k-- > 0;) group_start[group[order[k]]] = k;
    auto fail = [&](int rc, const char* what) {
        if (rc != SWB_OK) throw MarlinError(std::string(what) + ": " + swb_last_error(c));
    };
    // the two sides of each group's equation: (sum rho A, h), (-sum rho B, beta_h)
    auto sums = [&](size_t lo, size_t hi) {
        std::vector<std::pair<G1Point, G2Point>> pairs;
        for (size_t g = 0; g < group_key.size(); g++) {
            const size_t a = std::max(lo, group_start[g]), e = std::min(hi, group_start[g + 1]);
            if (a >= e || live_before[e] == live_before[a]) continue;
            // the MSMs run over the whole bucket range whatever the context's bucket shard: a share would be useless here
            const BucketShard whole{0, 1};
            size_t ida, idb;
            fail(msm_queue_submit(c, &bases, base[a], sc_dev + base[a], base[e] - base[a], 1, whole, &ida), "verify_batch: msm");
            fail(msm_queue_submit(c, &bases, base[a], sc_dev + total + base[a], base[e] - base[a], 1, whole, &idb), "verify_batch: msm");
            fail(msm_queue_flush(c), "verify_batch: msm");
            Terms key;                                  // (on the host while the two MSMs run)
            for (size_t k = a; k < e; k++)
                if (bp[order[k]].live)
                    for (auto& t : bp[order[k]].key_terms) add_term(key, t.first, t.second);
            std::vector<std::pair<G1Point, Fr>> kv;
            for (auto& t : key) kv.push_back({*t.first, t.second});
            const G1Point key_part = to_affine(g1_msm_host(kv));
            swb_g1_jacobian ra, rb;
            fail(msm_queue_result(c, ida, &ra), "verify_batch: msm");
            fail(msm_queue_result(c, idb, &rb), "verify_batch: msm");
            pairs.push_back({g1_add(from_jacobian(ra), key_part), group_key[g]->h});
            pairs.push_back({g1_neg(from_jacobian(rb)), group_key[g]->beta_h});
        }
        return pairs;
    };
    auto holds = [&](size_t lo, size_t hi) {
        const auto pairs = sums(lo, hi);
        return pairs.empty() || pairing_product_is_one(pairs);
    };
    auto accept = [&](size_t lo, size_t hi) {
        for (size_t k = lo; k < hi; k++)
            if (bp[order[k]].live) ok[order[k]] = 1;
    };
    const auto all = sums(0, n);
    st.mark("msm");
    const bool all_hold = all.empty() || pairing_product_is_one(all);
    st.mark("pairing");
    if (all_hold) {
        accept(0, n);
    } else {
        // [lo, hi) is known to fail when known_bad; returns whether every live proof in it was accepted
        std::function<bool(size_t, size_t, bool)> decide = [&](size_t lo, size_t hi, bool known_bad) {
            const size_t cnt = live_before[hi] - live_before[lo];
            if (cnt == 0) return true;
            if (!known_bad && holds(lo, hi)) {
                accept(lo, hi);
                return true;
            }
            if (cnt == 1) return false;
            size_t mid = lo;
            while (live_before[mid] - live_before[lo] < cnt / 2) mid++;
            const bool left = decide(lo, mid, false);
            decide(mid, hi, left);      // the halves' equations multiply to the failing one: both cannot hold
            return false;
        };
        decide(0, n, true);
    }
    st.mark("bisect");
    return SWB_OK;
}

}  // namespace swb
