/* swb200 -- B200-native (sm_100a) backend for the Marlin prover hot path of lambdaclass/simpleworks.
 *
 * C ABI of libswb200.{a,so}: exactly what a Rust `extern "C"` block in a sibling FFI crate would
 * bind (simpleworks itself is #![forbid(unsafe_code)], reference src/lib.rs:2).  Plain pointers
 * and sizes only.  There is no plugin registry in simpleworks / arkworks 0.3 -- dispatch is by
 * static generics -- so each entry point names the upstream call shape it replaces and the
 * reference call site that reaches it:
 *
 *   swb_msm_g1*            ark_ec::msm::VariableBaseMSM::multi_scalar_mul(&[G1Affine], &[BigInteger256])
 *                          <- kzg10::commit/open <- MarlinKZG10::commit/open <- Marlin::index/prove
 *                          <- reference src/marlin/mod.rs:75,92; src/merkle_tree/simple_merkle_tree.rs:83,119
 *   swb_ntt_fr*            ark_poly::Radix2EvaluationDomain::{fft,ifft,coset_fft,coset_ifft}_in_place
 *                          <- AHP indexer + prover rounds <- reference src/marlin/mod.rs:75,92
 *   swb_fixed_base_powers  ark_ec::msm::FixedBaseMSM::{get_window_table,multi_scalar_mul} + batch
 *                          normalisation <- KZG10::setup <- Marlin::universal_setup
 *                          <- reference src/marlin/mod.rs:52; simple_merkle_tree.rs:39
 *   swb_fr_*, swb_fq_*     ark_ff::Fp256<FrParameters> / Fp384<FqParameters> arithmetic (vector forms)
 *
 * Data types are bit-identical to the arkworks in-memory representation (Montgomery form,
 * little-endian u64 limbs), so a Rust shim passes slices straight through (see INTEGRATION.md).
 *
 * Conventions: every call returns 0 on success or an SWB_E* class; text via swb_last_error().
 * The library never aborts and never falls back to the CPU: without a CUDA device swb_init
 * fails with SWB_ECUDA.  A swb_ctx owns one device and one stream; it is single-threaded (one
 * call in flight); several contexts (one per GPU / process) may coexist.  Pointers named *_host
 * are ordinary host memory borrowed for the duration of the call; *_dev are device pointers on
 * the context's device.
 */
#ifndef SWB200_H
#define SWB200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct { uint64_t l[4]; } swb_fr;        /* ark_ff::Fp256<FrParameters>, Montgomery   */
typedef struct { uint64_t l[4]; } swb_bigint256; /* ark_ff::BigInteger256, canonical integer  */
typedef struct { uint64_t l[6]; } swb_fq;        /* ark_ff::Fp384<FqParameters>, Montgomery   */
typedef struct { swb_fq x, y; uint8_t infinity; uint8_t _pad[7]; } swb_g1_affine;   /* 104 B  */
typedef struct { swb_fq x, y, z; } swb_g1_jacobian;                /* 144 B, (X/Z^2, Y/Z^3)    */

typedef struct swb_ctx swb_ctx;
typedef struct swb_bases swb_bases;

enum { SWB_OK = 0, SWB_ECUDA = 1, SWB_EARG = 2, SWB_ENOMEM = 3, SWB_EINTERNAL = 4 };

/* ---- context ---------------------------------------------------------------------------- */
int  swb_init(int device, swb_ctx** out);
void swb_destroy(swb_ctx*);
const char* swb_last_error(const swb_ctx*);
/* Hands back every device allocation the context only keeps for reuse: the scratch arenas of MSM / NTT / sort (they
 * grow to the largest call seen: 90 GB after a 2^26-point MSM), the cache of released vectors and the NTT twiddle
 * table.  Nothing a live handle owns is touched; the next call allocates again.  Waits for all work of the context
 * first; fails while an MSM begun with the asynchronous interface has not been collected. */
int  swb_trim(swb_ctx*);      /* NULL ctx -> last error of a failed swb_init */
/* run all work of this context on an existing CUDA stream (cudaStream_t), e.g. the caller's
 * current stream so that its events time the kernels and its later work is ordered after ours;
 * NULL is the CUDA legacy default stream.  swb_reset_stream returns to the context's own
 * (non-blocking) stream, which is what a fresh context uses. */
int  swb_set_stream(swb_ctx*, void* cuda_stream);
int  swb_reset_stream(swb_ctx*);
int  swb_sync(swb_ctx*);
int  swb_device_info(swb_ctx*, int* sm_count, int* cc_major, int* cc_minor, size_t* total_mem);
/* number of kernels this context has launched since creation (bench.py's gpu_launches) */
uint64_t swb_launch_count(const swb_ctx*);

/* ---- device buffers (thin cudaMalloc/cudaMemcpy wrappers so non-CUDA hosts can stay resident) */
int  swb_dev_alloc(swb_ctx*, size_t bytes, void** out_dev);
int  swb_dev_free(swb_ctx*, void* dev);
int  swb_h2d(swb_ctx*, void* dst_dev, const void* src_host, size_t bytes);
int  swb_d2h(swb_ctx*, void* dst_host, const void* src_dev, size_t bytes);

/* ---- field vectors: r[i] = a[i] op b[i]  (device pointers; parity + throughput probes) ---- */
int  swb_fr_mul_vec_dev(swb_ctx*, swb_fr* r_dev, const swb_fr* a_dev, const swb_fr* b_dev, size_t n);
int  swb_fr_add_vec_dev(swb_ctx*, swb_fr* r_dev, const swb_fr* a_dev, const swb_fr* b_dev, size_t n);
int  swb_fr_sub_vec_dev(swb_ctx*, swb_fr* r_dev, const swb_fr* a_dev, const swb_fr* b_dev, size_t n);
int  swb_fq_mul_vec_dev(swb_ctx*, swb_fq* r_dev, const swb_fq* a_dev, const swb_fq* b_dev, size_t n);
int  swb_fq_add_vec_dev(swb_ctx*, swb_fq* r_dev, const swb_fq* a_dev, const swb_fq* b_dev, size_t n);
int  swb_fq_sub_vec_dev(swb_ctx*, swb_fq* r_dev, const swb_fq* a_dev, const swb_fq* b_dev, size_t n);
/* ark_ff::batch_inversion (zeros stay zero), in place */
int  swb_fr_batch_inverse_dev(swb_ctx*, swb_fr* v_dev, size_t n);
/* Measures the achievable 32x32->64 multiply-accumulate ("limb-product") rate of this GPU with
 * a register-resident Montgomery-multiplication loop: the integer roofline denominator.
 * field: 0 = Fr (128 limb-products per multiplication), 1 = Fq (288).  Returns limb-products/s
 * and field multiplications/s measured with CUDA events. */
int  swb_measure_mul_peak(swb_ctx*, int field, int iters, double* limb_products_per_s, double* muls_per_s);

/* Raw integer-pipe probe: independent multiply-accumulate chains held in registers.
 * kind 0: 32-bit IMAD (mad.lo.u32), kind 1: 32x32+64 IMAD.WIDE (mad.wide.u32), kind 2: IMAD.WIDE.U32.X
 * carry chains of length four (mad.lo.cc / madc.hi.cc pairs), kind 3: IADD3.X add-with-carry
 * chains (ALU pipe).  ops/s by CUDA events. */
int  swb_measure_imad_peak(swb_ctx*, int kind, int iters, double* ops_per_s);

/* ---- per-stage timings of the last MSM / NTT call (CUDA events on the context's stream) ----- */
/* enable != 0 makes every later call record events at its stage boundaries (a few microseconds);
 * swb_profile_last copies up to cap (name, milliseconds) pairs of the most recent call.         */
int  swb_profile_enable(swb_ctx*, int enable);
int  swb_profile_last(swb_ctx*, const char** names, double* ms, int cap, int* count);

/* ---- G1 bases (SRS / committer key): upload once, keep resident --------------------------- */
int  swb_bases_load(swb_ctx*, const swb_g1_affine* host, size_t n, swb_bases** out);
/* same from a device buffer of swb_g1_affine (104-byte records) */
int  swb_bases_load_dev(swb_ctx*, const swb_g1_affine* dev, size_t n, swb_bases** out);
/* bases[i] = beta^i * g generated on the device and kept there (KZG10::setup's powers_of_g without
 * the round trip through the host) */
int  swb_bases_from_powers(swb_ctx*, const swb_g1_jacobian* g_host, const swb_fr* beta_host, size_t n, swb_bases** out);
/* copy n bases starting at offset back to the host as 104-byte GroupAffine records */
int  swb_bases_export(swb_ctx*, const swb_bases*, size_t offset, size_t n, swb_g1_affine* out_host);
/* Window tables: besides each base P_i keep 2^(c*j) * P_i for j < ceil(253 / c), so that MSMs over
 * these bases accumulate all windows into ONE set of 2^(c-1) buckets (one bucket reduction, no
 * doublings) and scalars above r/2 are replaced by r - s on the negated point, which saves the carry
 * window.  window_bits = 0 picks c from the number of bases.  Memory grows ceil(253/c)-fold.
 * Calling this asserts that every base lies in the prime-order subgroup (true for the KZG powers
 * beta^i * G that ark-poly-commit's kzg10::commit passes to VariableBaseMSM); results are then
 * identical to the plain path.  MSMs much smaller than the table (n * levels < 8 * 2^(c-1)) keep
 * using the plain path on level 0. */
int  swb_bases_precompute(swb_ctx*, swb_bases*, int window_bits);
/* window_bits / levels of the tables, both 0 when none were built */
int  swb_bases_table_info(const swb_bases*, int* window_bits, int* levels);
size_t swb_bases_len(const swb_bases*);
void swb_bases_free(swb_bases*);

/* ---- variable-base MSM: out = sum_{i<n} scalars[i] * bases[offset+i] ---------------------- */
/* Result is a Jacobian point with Z = 1 (or (0,1,0) for the identity): the unique affine value
 * arkworks' callers obtain after into_affine(), so results compare bit-for-bit.             */
int  swb_msm_g1(swb_ctx*, const swb_bases*, size_t offset, const swb_bigint256* scalars_host, size_t n,
                swb_g1_jacobian* out_host);
int  swb_msm_g1_dev(swb_ctx*, const swb_bases*, size_t offset, const swb_bigint256* scalars_dev, size_t n,
                    swb_g1_jacobian* out_host);
/* scalars given in Montgomery form (Fr), converted on the device -- what kzg10::commit does with
 * into_repr() on the host today */
int  swb_msm_g1_fr_dev(swb_ctx*, const swb_bases*, size_t offset, const swb_fr* scalars_dev, size_t n,
                       swb_g1_jacobian* out_host);
/* the same with host-resident Montgomery scalars (what a polynomial's coefficient vector is) */
int  swb_msm_g1_fr(swb_ctx*, const swb_bases*, size_t offset, const swb_fr* scalars_host, size_t n,
                   swb_g1_jacobian* out_host);
/* Multi-GPU proving.  One process per GPU runs the same prover on the same inputs (the protocol is
 * deterministic, so every rank holds every polynomial); after this call each commit / open MSM of
 * swb_marlin_index and swb_marlin_prove on this context only covers the rank's contiguous share of
 * the (base, scalar) index range and `combine` is called with the 144-byte partial result: it must
 * return the sum over all ranks (an all-gather of world x 144 bytes followed by swb_g1_sum_jacobian --
 * simpleworks_b200/binding.py does it with torch.distributed over NCCL).  Every rank then continues
 * with identical commitments, so the proof bytes are those of a single GPU.  world <= 1 switches it off; a NULL
 * callback uses the context's own communicator (swb_comm_init, below).  The callback returns 0 on success. */
typedef int (*swb_combine_fn)(void* user, const swb_g1_jacobian* mine, swb_g1_jacobian* sum);
int  swb_set_msm_shard(swb_ctx*, int rank, int world, swb_combine_fn combine, void* user);
/* Multi-GPU proving from one process.  The protocol calls on ctx (swb_marlin_index, swb_marlin_prove,
 * swb_pk_deserialize) share each commit / open MSM between ctx (rank 0) and the n_peers other contexts (ranks
 * 1..n_peers), in this process, on any devices, the same device included.  The split is swb_set_msm_shard's for a
 * world of 1 + n_peers: by bucket in a power-of-two world once the SRS powers have window tables, by index range
 * otherwise.  For every MSM the scalars a peer reads (all of them by bucket, its slice by index) are copied to its
 * device with cudaMemcpyPeerAsync (direct where the devices allow peer access, which this call enables for the
 * process, staged through the host elsewhere), the share runs on the peer's own stream and MSM slots, and ctx adds the
 * shares on the host.  The calling thread launches on every device and only waits for the results; the NTTs and
 * polynomial work stay on ctx.  Proof and key bytes are those of one GPU.  n_peers = 0 detaches.  Refused (SWB_EARG)
 * while ctx shards through swb_set_msm_shard or is itself a peer, for a peer that has peers or a shard of its own, for
 * ctx itself or a repeated peer, and while an MSM is in flight; swb_set_msm_shard in turn refuses ctx and its peers.
 * The peers plan their shares with ctx's MSM settings (swb_msm_set_window_bits, _set_table_policy, _set_pair_sums),
 * whatever their own are, so that all ranks decompose the scalars alike.
 * Lifetimes: the first sharded MSM over an SRS's powers copies them to every peer (replicas, which later receive the
 * SRS's window tables by copy too; a peer without room for the tables keeps that SRS's MSMs on index-range shares); the
 * SRS owns its replicas and frees them on the peer contexts when it is freed.  So the peers must outlive every SRS and
 * proving key created on ctx.  Contexts may then be destroyed in any order: swb_destroy of ctx or of a peer detaches
 * it from the other side.  A peer is busy while ctx's call runs: no other thread may use it then.  Not shared:
 * swb_marlin_verify_batch, the swb_msm_g1* calls, NTTs and polynomial work. */
int  swb_set_msm_peers(swb_ctx*, swb_ctx* const* peers, int n_peers);
/* bytes ctx has copied to its peers since it was created: SRS replicas and MSM scalars */
uint64_t swb_peer_copy_bytes(const swb_ctx*);
/* ---- multi-GPU exchange inside the library (one process per GPU; NCCL resolved at run time) ---------------
 * swb_comm_unique_id: rank 0 obtains the 128-byte ncclUniqueId and hands it to the other ranks out of band
 * (any channel: a file, MPI, torch.distributed's store); swb_comm_init: every rank joins, on its context's
 * device; swb_comm_sum_g1: out[k] = sum over all ranks of mine[k] for k < count -- ONE ncclAllGather of
 * world x count x 144 bytes on the context's stream, then host additions, identical on every rank.  With a
 * communicator in place swb_set_msm_shard may be called with a NULL callback: the prover's partial commitments
 * then travel through it, all MSMs of a prover round in one all-gather.  swb_destroy ends the communicator. */
int  swb_comm_unique_id(uint8_t id[128]);
int  swb_comm_init(swb_ctx*, const uint8_t id[128], int rank, int world);
int  swb_comm_info(const swb_ctx*, int* rank, int* world);
int  swb_comm_sum_g1(swb_ctx*, const swb_g1_jacobian* mine_host, size_t count, swb_g1_jacobian* out_host);
int  swb_comm_destroy(swb_ctx*);
/* n_msms independent MSMs over the same bases (the commitments of one prover round: ark-poly-commit's
 * `commit` loops over its polynomials): MSM i takes ns[i] device-resident scalars scalars_dev[i]
 * (canonical integers, or Montgomery values when montgomery != 0) against bases[offsets[i] ..] and writes
 * outs[i].  Over bases with window tables (swb_bases_precompute) up to 16 MSMs at a time run as ONE pipeline --
 * one digits pass, one sort with the vector index in the key's top bits, one accumulation, one bucket reduction
 * with a bucket set per vector -- so the per-MSM bucket tail and launch gaps are paid once per batch.  Otherwise
 * two MSMs are in flight at a time on streams of their own, which hides the latency-bound bucket reduction of
 * one under the accumulation of the next.  Results equal n_msms single calls either way. */
int  swb_msm_g1_batch_dev(swb_ctx*, const swb_bases*, const size_t* offsets, const void* const* scalars_dev, const size_t* ns,
                          size_t n_msms, int montgomery, swb_g1_jacobian* outs);
/* Bucket sharding over `world` GPUs (a power of two): every rank holds ALL bases and sees ALL scalars, but only
 * fills the buckets b with b mod world == rank of each bucket set (interleaved: equal load whatever the digit
 * distribution), so the window width -- and with
 * window tables the single shared bucket set -- stays what one GPU would use while sort, accumulation and bucket
 * reduction all shrink by `world` (index-range sharding cannot shrink the bucket reduction).  Every swb_msm_g1*
 * call on the context then returns this rank's share; the full result is the sum of the shares of all ranks
 * (swb_g1_sum_jacobian, or swb_comm_* below).  world <= 1 switches it off. */
int  swb_msm_set_bucket_shard(swb_ctx*, int rank, int world);
/* the signed-digit window width c and window count ceil(254/c) an n-point MSM will use */
int  swb_msm_plan(swb_ctx*, size_t n, int* window_bits, int* windows);
/* window width override for tuning/tests (0 = automatic) */
int  swb_msm_set_window_bits(swb_ctx*, int c);
/* Batch-affine pair sums: before the bucket accumulation, neighbouring sorted positions of the same bucket are added in
 * affine coordinates with one shared inversion per thread block (~6 field products per pair instead of the 10 of an
 * XYZZ mixed addition), then the sums of neighbouring pairs, and so on for up to four levels, so that the accumulation adds
 * one point per block of up to 16 positions.  1 = automatic (large MSMs with well-filled buckets; the default),
 * 0 = never, 2..5 = always, with 1..4 levels.  Results are identical. */
int  swb_msm_set_pair_sums(swb_ctx*, int policy);
/* which path MSMs over bases with window tables take: 0 = automatic (the rule above), 1 = the table
 * path whatever n is, -1 = the plain path on level 0.  Results are identical; tests and bench.py use it
 * to compare the two paths on the same input. */
int  swb_msm_set_table_policy(swb_ctx*, int policy);
/* sum of n Jacobian points on the host side of the ABI (combining per-GPU partial MSMs); pure
 * host arithmetic, ctx may be NULL */
int  swb_g1_sum_jacobian(swb_ctx*, const swb_g1_jacobian* pts_host, size_t n, swb_g1_jacobian* out_host);

/* ---- fixed-base: out[i] = beta^i * g, i < n, affine (KZG10::setup powers_of_g) ------------ */
int  swb_fixed_base_powers(swb_ctx*, const swb_g1_jacobian* g_host, const swb_fr* beta_host, size_t n,
                           swb_g1_affine* out_host);

/* ---- radix-2 NTT over Fr, natural order in and out, in place ------------------------------ */
/* inverse: uses w^-1 and scales by n^-1.  coset: multiplies by 22^j before a forward transform,
 * by 22^-j after an inverse one.  log_n <= 30 (Fr two-adicity is 47; bounded here by tables).
 * Inputs are Montgomery-form field elements below r, as every ark_ff Fr is; outputs are canonical again
 * (inside, the butterflies work in the lazy range [0, 2r)).  Transforms of more than one pass keep a table of
 * all powers of the root for the largest size seen (32 B << log_n, at most 2 GiB; swb_trim releases it). */
int  swb_ntt_fr(swb_ctx*, swb_fr* inout_host, uint32_t log_n, int inverse, int coset);
int  swb_ntt_fr_dev(swb_ctx*, swb_fr* inout_dev, uint32_t log_n, int inverse, int coset);
int  swb_ntt_fr_batch_dev(swb_ctx*, swb_fr* inout_dev, uint32_t log_n, size_t batch, int inverse, int coset);

/* ==== protocol level: simpleworks::marlin (reference src/marlin/mod.rs:33-94, serialization.rs) ====
 * Opaque handles and canonical bytes.  Host orchestration in C++ inside the library; all NTTs,
 * MSMs and fixed-base tables run on the GPU of the context.
 *   swb_rng_test_rng             generate_rand()  = ark_std::test_rng()            mod.rs:33-35
 *   swb_marlin_universal_setup   generate_universal_srs                             mod.rs:45-55
 *   swb_marlin_index             generate_proving_and_verifying_keys               mod.rs:88-94
 *   swb_marlin_prove             generate_proof + serialize_proof    mod.rs:70-77, serialization.rs:5
 *   swb_marlin_verify            deserialize_proof + verify_proof    serialization.rs:14, mod.rs:79-86
 *   swb_marlin_verify_batch      the same for many proofs at once (SimpleMerkleTree::verify, a ledger's block)
 * swb_r1cs is what a ConstraintSystemRef exposes (to_matrices() + assignments; mod.rs:16): columns
 * are instance variables first (column 0 = the constant one), then witnesses.  public_inputs for
 * verify exclude the leading one, as in simple_merkle_tree.rs:133-143.
 * An unsatisfied instance makes swb_marlin_prove fail (the reference panics through a
 * debug_assert, examples/schnorr-signature/main.rs:214-217).
 * Verification evaluates the KZG pairing-product check on the host (Fq2/Fq6/Fq12 tower, ate
 * pairing); the verifying key holds g, gamma_g, h, beta_h and the degree-bound shift powers, never
 * the trapdoor. */
typedef struct swb_rng swb_rng;
typedef struct swb_r1cs swb_r1cs;
typedef struct swb_srs swb_srs;
typedef struct swb_pk swb_pk;
typedef struct swb_vk swb_vk;

swb_rng* swb_rng_test_rng(void);
/* rand::rngs::StdRng::from_seed (ChaCha12 keyed with 32 bytes) and StdRng::from_entropy (seeded from the
 * operating system; NULL when no entropy source is available).  test_rng() is a PUBLIC fixed seed: it makes
 * setup's trapdoor, the prover's blinders and the verifier's batching scalar predictable, so outside tests use
 * one of these. */
swb_rng* swb_rng_from_seed(const uint8_t seed[32]);
swb_rng* swb_rng_from_entropy(void);
uint64_t swb_rng_next_u64(swb_rng*);
void swb_rng_free(swb_rng*);

swb_r1cs* swb_r1cs_new(size_t num_instance /* incl. the constant one */, size_t num_witness);
/* built-in instances: 0 manual-constraints (v0 = a, v1 = b), 1 test-circuit UInt8 equality
 * (v0, v1), 2 synthetic chain x_i * x_{i+1} = x_{i+2} with `size` constraints (v0, v1 = seeds),
 * 3 synthetic general-shape instance: `size` constraints, v0 random terms per row of A and B (columns
 * may repeat), 3 public inputs, seed v1 */
swb_r1cs* swb_r1cs_builtin(int kind, size_t size, uint64_t v0, uint64_t v1);
int  swb_r1cs_add_constraint(swb_r1cs*, const swb_fr* a_coef, const uint32_t* a_col, size_t na,
                             const swb_fr* b_coef, const uint32_t* b_col, size_t nb,
                             const swb_fr* c_coef, const uint32_t* c_col, size_t nc);
int  swb_r1cs_set_assignment(swb_r1cs*, const swb_fr* instance, size_t ni, const swb_fr* witness, size_t nw);
int  swb_r1cs_is_satisfied(const swb_r1cs*);
void swb_r1cs_free(swb_r1cs*);

/* Host-side phase times of the protocol calls (process-wide): after swb_marlin_profile_enable(1) every
 * swb_marlin_index / swb_marlin_prove leaves "<call>: phase=milliseconds ..." (wall-clock time the host
 * spent in each phase -- msm and ntt are nested inside the round phases; GPU work is asynchronous, so a
 * phase also pays for what was queued before it) for swb_marlin_last_phases, which copies at most cap
 * bytes including the terminator and returns the size needed. */
int    swb_marlin_profile_enable(int enable);
size_t swb_marlin_last_phases(char* buf, size_t cap);
int  swb_marlin_universal_setup(swb_ctx*, size_t num_constraints, size_t num_variables, size_t num_non_zero,
                                swb_rng*, swb_srs** out);
size_t swb_srs_max_degree(const swb_srs*);
/* The SRS counts the commit/open MSMs it serves; after n_msms of them its powers get window tables
 * (swb_bases_precompute, digit width chosen for the MSM sizes seen so far) so that later commitments
 * run on the single-bucket-set path (about 13 % faster proofs; building the tables costs about four
 * proofs).  Default 400, i.e. some twenty proofs (SWB_MARLIN_TABLES overrides), 0 = never, 1 = at the
 * first commitment.  Proof bytes do not depend on it. */
int  swb_srs_set_tune_after(swb_srs*, long n_msms);
/* window tables of the SRS powers: digit width and number of levels, both 0 while the plain path is in use (the
 * tables are skipped when they would not fit in half of the free device memory). */
int  swb_srs_table_info(const swb_srs*, int* window_bits, int* levels);
/* Handle lifetimes: a proving key keeps its SRS alive (reference counted), so swb_srs_free and swb_pk_free
 * may come in either order; every SRS, proving key and bases handle must be freed BEFORE swb_destroy of the
 * context it was created on, and is only valid on that context (other contexts are refused with SWB_EARG). */
void swb_srs_free(swb_srs*);
int  swb_marlin_index(swb_ctx*, const swb_srs*, const swb_r1cs*, swb_pk** pk, swb_vk** vk);
void swb_pk_free(swb_pk*);
void swb_vk_free(swb_vk*);
int  swb_marlin_prove(swb_ctx*, const swb_pk*, const swb_r1cs* cs_with_assignment, swb_rng*, uint8_t** proof, size_t* len);
/* rng supplies the scalar that folds the two opening equations into one pairing product (the
 * reference passes its StdRng, mod.rs:79-86).  The scalar must be unpredictable to the prover -- the
 * opening proofs are not bound by the transcript -- so NULL draws it from OS entropy, never from a fixed
 * seed.  ctx may be NULL: verification is host arithmetic (BLS12-377 pairing), no GPU involved. */
int  swb_marlin_verify(swb_ctx*, const swb_vk*, const swb_fr* public_inputs, size_t n, const uint8_t* proof, size_t len,
                       swb_rng*, int* ok);
/* Verifies n proofs in one call: ok[i] = the verdict of swb_marlin_verify(ctx, vks[i], public_inputs[i], n_inputs[i],
 * proofs[i], lens[i]) for every i < n, except with negligible probability; proofs and keys as in swb_marlin_verify.
 * A malformed proof, a point off the curve or outside G1, a wrong input count or a missing shift power gives ok[i] = 0,
 * not an error.  The keys may all be the same or all differ; proofs whose keys share (h, beta_h) -- keys indexed from
 * one SRS -- are checked together by ONE pairing equation, the proofs weighted by independent secret 128-bit scalars;
 * when it fails, halves of the proofs are checked the same way until each invalid proof is found.  The context is
 * required: the proofs' G1 points are decoded and summed (MSM) on its GPU; the context's bucket shard does not apply.
 * rng as in swb_marlin_verify (NULL: OS entropy, never a fixed seed).  The call draws 2 n u128 from it: for each proof
 * in index order, whether or not it parses, its weight and then the scalar that folds its two openings, so a seeded
 * rng gives reproducible verdicts.  Returns non-zero only for bad arguments, CUDA failures or a missing entropy
 * source, and then every ok[i] is 0; n = 0 returns SWB_OK.  With swb_profile_enable the stage times (parse, decode,
 * transcripts, msm, pairing, bisect) are kept for swb_profile_last. */
int  swb_marlin_verify_batch(swb_ctx*, size_t n, const swb_vk* const* vks, const swb_fr* const* public_inputs,
                             const size_t* n_inputs, const uint8_t* const* proofs, const size_t* lens, swb_rng*, int* ok);
void swb_bytes_free(uint8_t*);
/* serialize_verifying_key / deserialize_verifying_key (reference src/marlin/serialization.rs:19-31);
 * NULL on malformed input. */
int  swb_vk_serialize(const swb_vk*, uint8_t** bytes, size_t* len);
swb_vk* swb_vk_deserialize(const uint8_t* bytes, size_t len);
/* deserialize_proof / serialize_proof as objects (serialization.rs:5-17): NULL unless the bytes are a canonical
 * proof (every point on the curve, in the subgroup, coordinates and scalars reduced, nothing trailing);
 * swb_marlin_verify_proof = verify_proof on the object (mod.rs:79-86). */
typedef struct swb_proof swb_proof;
swb_proof* swb_proof_deserialize(const uint8_t* bytes, size_t len);
int  swb_proof_serialize(const swb_proof*, uint8_t** bytes, size_t* len);
void swb_proof_free(swb_proof*);
int  swb_marlin_verify_proof(swb_ctx*, const swb_vk*, const swb_fr* public_inputs, size_t n, const swb_proof*, swb_rng*, int* ok);
/* serialize_proving_key / deserialize_proving_key (serialization.rs:33-45).  Like upstream's, the bytes carry the
 * committer key (all SRS powers up to max_degree, 96 bytes each) next to the constraint matrices, so a key loads
 * without the SRS it was indexed from; the layout ("SWBPK001", csrc/marlin_abi.cu) is this library's own.  Loading
 * re-derives the index on the device and fails unless it reproduces the verifying key stored in the bytes, which
 * is returned through vk (may be NULL). */
int  swb_pk_serialize(swb_ctx*, const swb_pk*, const swb_vk*, uint8_t** bytes, size_t* len);
int  swb_pk_deserialize(swb_ctx*, const uint8_t* bytes, size_t len, swb_pk** pk, swb_vk** vk);
/* R1CS interchange ("SWBR1CS1", layout in csrc/marlin/r1cs.hpp and INTEGRATION.md): constraint
 * systems synthesised by the reference's Rust gadgets, exported from ConstraintSystemRef */
swb_r1cs* swb_r1cs_read(const uint8_t* bytes, size_t len);
int  swb_r1cs_write(const swb_r1cs*, uint8_t** bytes, size_t* len);

#ifdef __cplusplus
}
#endif
#endif /* SWB200_H */
