// Engine-generic glue between the protocol templates (marlin.hpp) and a C ABI.  libswb200
// instantiates it with the CUDA engine (marlin_abi.cu -> swb_marlin_*), the oracle build with the
// CPU engine (oracle/marlin_oracle.cpp -> orc_marlin_*).  setup binds an engine to the SRS it makes;
// index and prove run on that SRS's engine.
#pragma once
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <random>
#include <string>

#include "marlin.hpp"

namespace swb {
namespace marlin {

struct RngHandle {
    ChaChaRng rng;
};
struct R1csHandle {
    R1cs cs;
};
template <class Engine>
struct SrsHandle {
    std::unique_ptr<UniversalSrs<Engine>> srs;
};
template <class Engine>
struct PkHandle {
    ProvingKey<Engine> pk;
};
struct VkHandle {
    VerifyingKey vk;
};

// StdRng::from_entropy(): 32 seed bytes from the operating system (/dev/urandom, std::random_device as a
// second source); false when neither is available
inline bool os_entropy(uint8_t seed[32]) {
    bool ok = false;
    if (FILE* f = fopen("/dev/urandom", "rb")) {
        ok = fread(seed, 1, 32, f) == 32;
        fclose(f);
    }
    if (!ok) {
        try {
            std::random_device rd;
            for (int i = 0; i < 8; i++) {
                const uint32_t w = rd();
                memcpy(seed + 4 * i, &w, 4);
            }
            ok = true;
        } catch (...) {
            ok = false;
        }
    }
    return ok;
}
inline RngHandle* rng_from_seed(const uint8_t seed[32]) {          // StdRng::from_seed = ChaCha12
    auto* h = new RngHandle();
    h->rng = ChaChaRng(seed, 12);
    return h;
}
inline RngHandle* rng_from_entropy() {
    uint8_t seed[32];
    if (!os_entropy(seed)) return nullptr;
    return rng_from_seed(seed);
}

inline Fr fr_from_abi(const uint64_t l[4]) {
    Fr r;
    for (int i = 0; i < 4; i++) { r.l[2 * i] = (uint32_t)l[i]; r.l[2 * i + 1] = (uint32_t)(l[i] >> 32); }
    return r;
}

inline R1csHandle* r1cs_new(size_t num_instance, size_t num_witness) {
    auto* h = new R1csHandle();
    h->cs.num_instance = num_instance ? num_instance : 1;
    h->cs.num_witness = num_witness;
    return h;
}
// one constraint <a, z> * <b, z> = <c, z>; coefficients are Montgomery Fr (4 x u64 each)
inline int r1cs_add_constraint(R1csHandle* h, const uint64_t* a_coef, const uint32_t* a_col, size_t na, const uint64_t* b_coef,
                               const uint32_t* b_col, size_t nb, const uint64_t* c_coef, const uint32_t* c_col, size_t nc) {
    const size_t nv = h->cs.num_variables();
    auto fill = [&](SparseRow& row, const uint64_t* coef, const uint32_t* col, size_t n) {
        for (size_t i = 0; i < n; i++) {
            if (col[i] >= nv) return false;
            row.e.push_back({fr_from_abi(coef + 4 * i), col[i]});
        }
        return true;
    };
    SparseRow ra, rb, rc;
    if (!fill(ra, a_coef, a_col, na) || !fill(rb, b_coef, b_col, nb) || !fill(rc, c_coef, c_col, nc)) return 1;
    h->cs.a.push_back(ra);
    h->cs.b.push_back(rb);
    h->cs.c.push_back(rc);
    return 0;
}
inline int r1cs_set_assignment(R1csHandle* h, const uint64_t* instance, size_t ni, const uint64_t* witness, size_t nw) {
    if (ni != h->cs.num_instance || nw != h->cs.num_witness) return 1;
    h->cs.instance.resize(ni);
    h->cs.witness.resize(nw);
    for (size_t i = 0; i < ni; i++) h->cs.instance[i] = fr_from_abi(instance + 4 * i);
    for (size_t i = 0; i < nw; i++) h->cs.witness[i] = fr_from_abi(witness + 4 * i);
    h->cs.has_assignment = true;
    return 0;
}
inline R1csHandle* r1cs_builtin(int kind, size_t size, uint64_t v0, uint64_t v1) {
    auto* h = new R1csHandle();
    switch (kind) {
        case 0: h->cs = circuit_manual_constraints(v0, v1); break;
        case 1: h->cs = circuit_uint8_equality((uint8_t)v0, (uint8_t)v1); break;
        case 2: h->cs = circuit_mul_chain(size, v0, v1); break;
        case 3: h->cs = circuit_random_sparse(size, v0, v1); break;
        default: delete h; return nullptr;
    }
    return h;
}

inline uint8_t* bytes_out(const std::vector<uint8_t>& b, size_t* len) {
    uint8_t* p = (uint8_t*)malloc(b.size() ? b.size() : 1);
    memcpy(p, b.data(), b.size());
    *len = b.size();
    return p;
}
// the parsers never let an exception (std::bad_alloc on hostile sizes included) cross the C boundary
inline R1csHandle* r1cs_from_bytes(const uint8_t* p, size_t len) {
    R1csHandle* h = nullptr;
    try {
        h = new R1csHandle();
        if (!r1cs_read(p, len, &h->cs)) { delete h; return nullptr; }
        return h;
    } catch (...) {
        delete h;
        return nullptr;
    }
}
inline uint8_t* r1cs_to_bytes(const R1csHandle* h, size_t* len) {
    std::vector<uint8_t> b;
    r1cs_write(h->cs, &b);
    return bytes_out(b, len);
}
inline uint8_t* vk_to_bytes(const VkHandle* vk, size_t* len) { return bytes_out(vk->vk.serialize(), len); }
inline VkHandle* vk_from_bytes(const uint8_t* p, size_t len) {
    VkHandle* h = nullptr;
    try {
        h = new VkHandle();
        if (!VerifyingKey::deserialize(p, len, &h->vk)) { delete h; return nullptr; }
        return h;
    } catch (...) {
        delete h;
        return nullptr;
    }
}

template <class Engine>
struct MarlinApi {
    static int setup(Engine& eng, size_t nc, size_t nv, size_t nnz, RngHandle* rng, SrsHandle<Engine>** out, std::string* err) {
        try {
            auto* h = new SrsHandle<Engine>();
            h->srs = universal_setup(eng, nc, nv, nnz, rng->rng);
            *out = h;
            return 0;
        } catch (const std::exception& e) {
            *err = e.what();
            return 4;
        }
    }
    static int index(const SrsHandle<Engine>* srs, const R1csHandle* cs, PkHandle<Engine>** pk, VkHandle** vk, std::string* err) {
        try {
            std::unique_ptr<PkHandle<Engine>> p(new PkHandle<Engine>());     // a key that fails mid-index is freed
            std::unique_ptr<VkHandle> v(new VkHandle());
            marlin::index(*srs->srs, cs->cs, &p->pk, &v->vk);
            host_profile().report("index");
            *pk = p.release();
            *vk = v.release();
            return 0;
        } catch (const std::exception& e) {
            *err = e.what();
            return 4;
        }
    }
    static int prove(const PkHandle<Engine>* pk, const R1csHandle* cs, RngHandle* rng, uint8_t** bytes, size_t* len, std::string* err) {
        try {
            Proof pr = marlin::prove(pk->pk, cs->cs, rng->rng);
            host_profile().report("prove");
            std::vector<uint8_t> b = pr.serialize();
            *bytes = (uint8_t*)malloc(b.size());
            memcpy(*bytes, b.data(), b.size());
            *len = b.size();
            return 0;
        } catch (const std::exception& e) {
            *err = e.what();
            return 4;
        }
    }
    // rng supplies the scalar that folds the two opening equations into one pairing product.  It MUST be
    // unpredictable to the prover: the opening proofs are not part of the transcript, so with a known scalar
    // two wrong equations can be made to cancel.  A null rng therefore draws from OS entropy (never from a
    // fixed seed); callers that want reproducible verification pass their own.
    static int verify(const VkHandle* vk, const uint64_t* public_inputs, size_t n, const uint8_t* proof, size_t len, RngHandle* rng,
                      int* ok, std::string* err) {
        try {
            Proof pr;
            *ok = 0;
            if (!Proof::deserialize(proof, len, &pr)) return 0;      // malformed proof: rejected, not an error
            std::vector<Fr> pi(n);
            for (size_t i = 0; i < n; i++) pi[i] = fr_from_abi(public_inputs + 4 * i);
            ChaChaRng local;
            if (!rng) {
                uint8_t seed[32];
                if (!os_entropy(seed)) { *err = "verify: no rng given and no OS entropy source available"; return 4; }
                local = ChaChaRng(seed, 12);
            }
            *ok = marlin::verify(vk->vk, pi, pr, rng ? rng->rng : local) ? 1 : 0;
            return 0;
        } catch (const std::exception& e) {
            *err = e.what();
            return 4;
        }
    }
};

}  // namespace marlin
}  // namespace swb
