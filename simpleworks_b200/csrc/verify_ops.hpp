// Batch verification of Marlin proofs (verify_ops.cu): the proofs' G1 points decoded on the GPU, one folded KZG
// pairing check per batch, bisection to find the invalid proofs.
#pragma once
#include "ctx.hpp"
#include "g1_decode.cuh"
#include "marlin/marlin.hpp"

namespace swb {

// status[i] and the swb_bases record (xy[2 i], xy[2 i + 1]) = g1_decode of the compressed encoding enc[12 i .. 12 i + 11]
// (48 bytes as little-endian words), for i < n; device pointers, enqueued on the context's stream
int g1_decode_dev(swb_ctx* c, const uint32_t* enc_dev, size_t n, const G1DecodeConsts& k, Fq* xy_dev, uint8_t* status_dev);

// ok[i] = the verdict of marlin::verify(*vks[i], public_inputs[i] (n_inputs[i] Montgomery Fr of 4 u64), proof i) for every
// i < n, except with negligible probability.  Draws 2 n u128 from rng: for proof i, in index order and whether or not it
// parses, its weight rho_i and then the scalar that folds its two openings.  The caller has set every ok[i] to 0.
// Stage times (parse, decode, transcripts, msm, pairing, bisect) go to the context's profile.
int marlin_verify_batch(swb_ctx* c, size_t n, const marlin::VerifyingKey* const* vks, const uint64_t* const* public_inputs,
                        const size_t* n_inputs, const uint8_t* const* proofs, const size_t* lens, marlin::ChaChaRng& rng, int* ok);

}  // namespace swb
