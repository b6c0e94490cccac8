/*
 * lurk_b200.h -- C ABI of liblurk_b200.so: the B200 (sm_100a) implementation of lurk-beta's Nova/SuperNova
 * proving hot path (SURVEY.md section 8).  Plain pointers and sizes only; no C++/torch types.
 *
 * The reference (argumentcomputer/lurk-beta @ f238d85c) has no FFI of its own: GPU work is delegated to
 * third-party crates via `--features cuda = ["neptune/cuda", "nova/cuda"]` (Cargo.toml:105-110).  Each entry
 * point below names the Rust seam it sits behind (reference file:line); INTEGRATION.md shows the
 * `extern "C"` binding a maintainer adds on the Rust side.
 *
 * Conventions
 *   - Field element: 32 bytes little-endian.  LURK_FMT_CANONICAL = the integer < p, i.e.
 *     ff::PrimeField::to_repr (src/field.rs:72-81).  LURK_FMT_MONTGOMERY = x * 2^256 mod p as 4 x u64, the
 *     in-memory form of pasta_curves (feature repr-c, Cargo.toml:42) and halo2curves field types, so Rust
 *     slices of `F` can be passed without conversion.
 *   - Affine point: x | y (64 bytes); the identity is (0, 0).  Result point: x | y | z (96 bytes) with
 *     z = 1 (finite) or x = y = z = 0 (identity), in the format asked for.
 *   - Ownership: the caller owns every buffer.  Contexts are created/destroyed by paired calls.
 *   - Errors: 0 = LURK_OK, negative = error; lurk_last_error() returns a thread-local message.  The library
 *     never aborts or unwinds (reference error style: Result<_, ProofError>, src/error.rs:8-18).
 *   - Threading: every call is re-entrant; `*_dev` calls are asynchronous on the given CUDA stream
 *     (a cudaStream_t passed as void*; NULL = default stream), host-buffer calls synchronise before returning.
 *   - Non-canonical inputs (>= p) are rejected with LURK_ERR_RANGE by the host-buffer calls (mirrors
 *     from_repr failing, src/field.rs:76-81); `*_dev` calls assume reduced inputs.
 *   - There is no CPU fallback: without a CUDA device every compute call returns LURK_ERR_NOGPU.
 */
#ifndef LURK_B200_H
#define LURK_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* LanguageField (src/field.rs:40-50) */
#define LURK_FIELD_BN254_FR 0  /* LanguageField::BN256   = halo2curves::bn256::Fr  (default, all benches) */
#define LURK_FIELD_BN254_FQ 1  /* LanguageField::Grumpkin = grumpkin::Fr = bn256::Fq                       */
#define LURK_FIELD_PALLAS_FQ 2 /* LanguageField::Pallas  = pallas::Scalar                                  */
#define LURK_FIELD_PALLAS_FP 3 /* LanguageField::Vesta   = vesta::Scalar = pallas::Base                    */

/* curves of the Nova curve cycles (src/proof/nova.rs:57-71) */
#define LURK_CURVE_BN254_G1 0 /* base Fq(1), scalars Fr(0) */
#define LURK_CURVE_GRUMPKIN 1 /* base Fr(0), scalars Fq(1) */
#define LURK_CURVE_PALLAS 2   /* base Fp(3), scalars Fq(2) */
#define LURK_CURVE_VESTA 3    /* base Fq(2), scalars Fp(3) */

#define LURK_FMT_CANONICAL 0
#define LURK_FMT_MONTGOMERY 1

#define LURK_OK 0
#define LURK_ERR_ARG (-1)
#define LURK_ERR_CUDA (-2)
#define LURK_ERR_OOM (-3)
#define LURK_ERR_RANGE (-4)
#define LURK_ERR_NOGPU (-5)
#define LURK_ERR_ORDER (-6) /* DAG nodes not topologically ordered */

const char *lurk_last_error(void);
int lurk_version(void);
int lurk_device_count(void);
/* modulus of a field as 32 bytes LE */
int lurk_field_modulus(int field_id, uint8_t out[32]);

/* ---------------------------------------------------------------------------------------------------
 * S1  Poseidon digests.  Replaces PoseidonCache::hash3/hash4/hash6/hash8 = neptune
 *     Poseidon::new_with_preimage(..).hash() (src/hash.rs:180-203) for a batch of independent preimages.
 *     arity in {3,4,6,8}; preimages n*arity elements, digests n elements.
 * ------------------------------------------------------------------------------------------------- */
int lurk_poseidon_hash_batch(int field_id, int arity, const uint8_t *preimages, size_t n, uint8_t *digests);
int lurk_poseidon_hash_batch_mont(int field_id, int arity, const uint8_t *preimages, size_t n, uint8_t *digests);
int lurk_poseidon_hash_batch_dev(int field_id, int arity, const void *d_preimages, size_t n, void *d_digests,
                                 int fmt, void *stream);
/* Constants as PoseidonConstants::new() builds them (src/hash.rs:61-72): R_F, R_P, the t*(R_F+R_P) round
 * constants and the t*t MDS matrix (row-major), canonical form.  Buffers may be NULL to query sizes. */
int lurk_poseidon_constants(int field_id, int arity, int *full_rounds, int *partial_rounds,
                            uint8_t *round_constants, uint8_t *mds);

/* ---------------------------------------------------------------------------------------------------
 * S3  Slot witnesses.  Replaces the per-slot body of generate_slots_witnesses (src/lem/multiframe.rs:520-592):
 *     allocate_slot -> neptune circuit2 poseidon_hash_allocated in witness mode (src/lem/circuit.rs:212-315).
 *     Output block per slot = [preimage (arity) | 3 aux per S-box in Neptune's optimised-round order | digest],
 *     lurk_poseidon_witness_block() elements (= hashN_cost + N, src/lem/multiframe.rs:503-516).
 *     Bit-decomposition slots: [value | aux of AllocatedNum::to_bits_le_strict] (src/lem/circuit.rs:241-243),
 *     lurk_bitdecomp_witness_block() elements (= BIT_DECOMP_*_WITNESS_SIZE, src/lem/multiframe.rs:495-498).
 * ------------------------------------------------------------------------------------------------- */
size_t lurk_poseidon_witness_block(int field_id, int arity);
int lurk_poseidon_witness_batch(int field_id, int arity, const uint8_t *preimages, size_t n, uint8_t *blocks,
                                int fmt);
int lurk_poseidon_witness_batch_dev(int field_id, int arity, const void *d_preimages, size_t n, void *d_blocks,
                                    int fmt, void *stream);
/* In-place form for the step witness: block k is written at element offset d_offsets[k] (u64, device) of d_base.  In the
 * reference every frame's aux is [its slot blocks in slot order | LEM body aux] (synthesize_frames_parallel,
 * src/lem/multiframe.rs:635-712), so the blocks of one slot type are strided by the frame length (9119 on BN256). */
int lurk_poseidon_witness_scatter_dev(int field_id, int arity, const void *d_preimages, size_t n, void *d_base,
                                      const void *d_offsets, int fmt, void *stream);
int lurk_bitdecomp_witness_scatter_dev(int field_id, const void *d_values, size_t n, void *d_base, const void *d_offsets,
                                       int fmt, void *stream);
size_t lurk_bitdecomp_witness_block(int field_id);
int lurk_bitdecomp_witness_batch(int field_id, const uint8_t *values, size_t n, uint8_t *blocks, int fmt);
int lurk_bitdecomp_witness_batch_dev(int field_id, const void *d_values, size_t n, void *d_blocks, int fmt,
                                     void *stream);

/* ---------------------------------------------------------------------------------------------------
 * S2  DAG hydration.  Replaces StoreCore::hydrate_z_cache / hash_ptr_val_unsafe (src/lem/store_core.rs:199-269)
 *     with the preimage layouts of `impl StoreHasher for PoseidonCache` (src/lem/store.rs:29-78).
 *     child[i] < n_atoms refers to atom digest child[i]; otherwise to node (child[i] - n_atoms), which must
 *     precede the referring node (children first).  out_digests: n elements, canonical.
 * ------------------------------------------------------------------------------------------------- */
#define LURK_DAG_TUPLE2 2     /* H4 [t0, d0, t1, d1]                 hash_ptrs len 2 (store.rs:31-36)  */
#define LURK_DAG_TUPLE3 3     /* H6                                   hash_ptrs len 3 (store.rs:37-50)  */
#define LURK_DAG_TUPLE4 4     /* H8                                   hash_ptrs len 4 (store.rs:51-67)  */
#define LURK_DAG_COMPACT 5    /* H4 [d0, t1, d1, d2]                  hash_compact    (store.rs:75-77)  */
#define LURK_DAG_COMMITMENT 6 /* H3 [d0 = secret, t1, d1]            hash_commitment (store.rs:70-73)  */
typedef struct lurk_dag_node {
    uint8_t kind;
    uint8_t reserved;
    uint16_t tag[4];   /* Tag::to_field = F::from(u16) (src/tag.rs:99-101) */
    uint32_t child[4];
} lurk_dag_node;
int lurk_dag_hash(int field_id, const lurk_dag_node *nodes, size_t n, const uint8_t *atom_digests,
                  size_t n_atoms, uint8_t *out_digests);
/* Routing aid, host only (works without a GPU): shape of the dependency DAG and a cost estimate.  A level costs one
 * dependent Poseidon latency on the GPU whatever its width, so deep and narrow stores (lists hashed cons by cons) are
 * faster on the caller's own CPU path (hash_ptr_val_unsafe, src/lem/store_core.rs:199-248), wide ones on the GPU.  The
 * library never hashes on the CPU itself: use_gpu == 0 means "keep this hydration on the reference's CPU path". */
typedef struct lurk_dag_plan {
    uint64_t nodes, levels, max_width;
    uint64_t est_gpu_us;       /* levels * ~170 us + nodes / 23 M/s + transfers */
    uint64_t est_cpu_core_us;  /* nodes * ~50 us on one core */
    int use_gpu;               /* est_gpu_us < the level-parallel CPU estimate on 8 cores */
} lurk_dag_plan;
int lurk_dag_hash_plan(const lurk_dag_node *nodes, size_t n, size_t n_atoms, lurk_dag_plan *plan);

/* ---------------------------------------------------------------------------------------------------
 * S4  Pedersen commitment = multi-scalar multiplication.  Replaces Arecibo
 *     CommitmentEngineTrait::commit -> DlogGroup::vartime_multiscalar_mul(scalars, bases) (called from
 *     RecursiveSNARK::prove_step, src/proof/nova.rs:287,292; supernova.rs:231-244).  The fixed commitment key
 *     is uploaded once into a context; each call streams scalars.
 * ------------------------------------------------------------------------------------------------- */
typedef struct lurk_msm_ctx lurk_msm_ctx;
/* bases_affine: n * 64 bytes, x || y per point, (0, 0) = identity.  Coordinates >= p or points off the curve are
 * rejected with LURK_ERR_RANGE (what the reference's point deserialisation checks before a key is used).  A context
 * belongs to the device that is current at creation; using it with another device current is LURK_ERR_ARG. */
int lurk_msm_ctx_create(int curve_id, const uint8_t *bases_affine, size_t n, int fmt, lurk_msm_ctx **out);
/* bases already on the current device (n * 64 bytes, Montgomery); the context borrows the pointer */
int lurk_msm_ctx_create_dev(int curve_id, const void *d_bases_mont, size_t n, lurk_msm_ctx **out);
void lurk_msm_ctx_destroy(lurk_msm_ctx *ctx);
/* curve and number of bases of a context (either output may be NULL) */
int lurk_msm_ctx_info(lurk_msm_ctx *ctx, int *curve_id, size_t *n);
/* sum_{i<n} scalars[i] * bases[i], n <= size of the key */
int lurk_msm_ctx_run(lurk_msm_ctx *ctx, const uint8_t *scalars, size_t n, int fmt, uint8_t out_xyz[96]);
int lurk_msm_ctx_run_dev(lurk_msm_ctx *ctx, const void *d_scalars, size_t n, int fmt, uint8_t out_xyz[96],
                         void *stream);
/* Fixed-base acceleration (the key never changes between folds): builds table[w][i] = 2^(c w) * bases[i] once
 * (nwin x n x 64 bytes of HBM; 1.7 GB for a 2^21-point key) so that all windows share one bucket set and a wider
 * window (c = 20) becomes affordable: ~13 instead of 16 bucket additions per scalar.  Results are unchanged.
 * Call before cloning; clones share the table. */
int lurk_msm_ctx_precompute(lurk_msm_ctx *ctx);
/* Asynchronous form: `launch` enqueues the whole commitment on `stream` and returns; `finish` waits for it and
 * produces the point.  One launch may be pending per context; `clone` gives another context on the same resident key
 * (own scratch; the parent must outlive it) so that e.g. commit(W) and commit(T) of one fold overlap. */
int lurk_msm_ctx_launch_dev(lurk_msm_ctx *ctx, const void *d_scalars, size_t n, int fmt, void *stream);
int lurk_msm_ctx_finish(lurk_msm_ctx *ctx, uint8_t out_xyz[96]);
int lurk_msm_ctx_clone(lurk_msm_ctx *ctx, lurk_msm_ctx **out);
/* Measurement hooks: when enabled, every run records CUDA events around the bucket-accumulation kernel (the dominant
 * kernel) on the launching stream; last_profile returns its duration and the number of kernels the run launched. */
int lurk_msm_ctx_set_profiling(lurk_msm_ctx *ctx, int enable);
int lurk_msm_ctx_last_profile(lurk_msm_ctx *ctx, float *accumulate_ms, unsigned *kernel_launches);
/* one-shot convenience (uploads bases every call) */
int lurk_msm(int curve_id, const uint8_t *bases_affine, const uint8_t *scalars, size_t n, int fmt,
             uint8_t out_xyz[96]);
/* Synthetic commitment key: bases_out[i] = [start + i + 1] G for the curve's standard generator, affine, n * 64 bytes
 * (host, multi-threaded).  The reference derives its key by hash-to-curve / powers of tau inside Arecibo
 * (public_params, src/proof/nova.rs:196-216) -- out of scope; this gives benches and tests a deterministic key of
 * distinct points (SURVEY.md 8(d) config 3). */
int lurk_synthetic_bases(int curve_id, uint64_t start, size_t n, int fmt, uint8_t *bases_out);
/* host-side sum of `count` result points (the per-GPU partial sums of a sharded commitment key) */
int lurk_point_sum(int curve_id, const uint8_t *points_xyz, size_t count, int fmt, uint8_t out_xyz[96]);

/* ---------------------------------------------------------------------------------------------------
 * N3  Commitment-key generation.  Replaces what `public_params` (src/proof/nova.rs:196-216, supernova.rs:117-137; cached on
 *     disk by src/public_parameters/mod.rs:20-71 because it takes minutes on the CPU) makes Arecibo do for the Pedersen key:
 *     R1CSShape::commitment_key -> CommitmentKey::setup(b"ck", n), n = next_power_of_two(max(#cons, #vars, ck_floor)) ->
 *     DlogGroup::from_label(label, n):  uniform_i = next 32 bytes of SHAKE256(label);
 *     G_i = Curve::hash_to_curve("from_uniform_bytes")(uniform_i), affine.
 *     hash_to_curve = halo2curves 0.6 (BN254 G1 / Grumpkin: BLAKE2b expand_message_xmd + Shallue-van de Woestijne, RFC 9380)
 *     or pasta_curves 0.5 (Pallas / Vesta: same hash_to_field + simplified SWU on the 3-isogenous curve + isogeny).
 *     The XOF is sequential and stays on a host thread, pipelined against the kernel that maps the points.
 * ------------------------------------------------------------------------------------------------- */
/* next_power_of_two(max(num_cons, num_vars, ck_floor)): the key length public_params asks for.  Host only. */
size_t lurk_ck_size(size_t num_cons, size_t num_vars, size_t ck_floor);
/* from_label: n affine points x | y (64 bytes each, identity = (0, 0)) in `fmt`. */
int lurk_ck_generate(int curve_id, const uint8_t *label, size_t label_len, size_t n, int fmt, uint8_t *bases_out);
/* same, written to device memory in Montgomery form -- exactly what lurk_msm_ctx_create_dev borrows: the key never crosses
 * PCIe.  Returns when the key is complete (the host thread feeds the XOF stream while the GPU works). */
int lurk_ck_generate_dev(int curve_id, const uint8_t *label, size_t label_len, size_t n, void *d_bases_mont, void *stream);
/* points first .. first + n - 1 of the same key: a rank's contiguous slice of a key sharded over GPUs (SURVEY.md 8(e)) */
int lurk_ck_generate_range_dev(int curve_id, const uint8_t *label, size_t label_len, size_t first, size_t n, void *d_bases_mont,
                               void *stream);
/* Curve::hash_to_curve(domain_prefix)(message) for n messages of msg_len bytes each (msg_len <= 64 and
 * msg_len + strlen(domain_prefix) <= ~80: everything must fit the single-block layout, else LURK_ERR_ARG). */
int lurk_hash_to_curve_batch(int curve_id, const char *domain_prefix, const uint8_t *messages, size_t msg_len, size_t n, int fmt,
                             uint8_t *points_out);
int lurk_hash_to_curve_batch_dev(int curve_id, const char *domain_prefix, const void *d_messages, size_t msg_len, size_t n,
                                 void *d_points, int fmt, void *stream);
/* Powers-of-tau key of the KZG engine (Arecibo hyperkzg CommitmentKey::setup -> UniversalKZGParam::gen_srs_for_testing; the
 * primary circuit's engine on BN256, src/proof/nova.rs:65-71): d_bases_mont[i] = beta^i * g for i < n, affine Montgomery, by
 * fixed-base windows of g.  g (64 bytes affine) and beta (32 bytes, scalar field) in `fmt`; how the reference derives them from
 * the label (a seeded RNG) and the verifier key's G2 side stay on the caller's CPU. */
int lurk_ck_powers_dev(int curve_id, const uint8_t g[64], const uint8_t beta[32], size_t n, void *d_bases_mont, int fmt, void *stream);
/* SHAKE256(in) -> out_len bytes (FIPS 202).  Host only (works without a GPU); the XOF behind from_label. */
int lurk_shake256(const uint8_t *in, size_t in_len, uint8_t *out, size_t out_len);

/* ---------------------------------------------------------------------------------------------------
 * N4  The data-parallel loops of `compress` (src/proof/nova.rs:341-356, supernova.rs:293-317 -> Arecibo CompressedSNARK::prove ->
 *     spartan::snark::RelaxedR1CSSNARK::prove): sum-check prover rounds over device-resident multilinear polynomials
 *     (SumcheckProof::prove_quad / prove_cubic_with_additive_term: compute_eval_points_* + bind_poly_var_top) and the folding rounds
 *     of the inner-product argument (provider::ipa_pc::InnerProductArgument::prove), the HyperKZG opening prover
 *     (provider::hyperkzg::EvaluationEngine::prove), plus EqPolynomial::evals and the inner product behind
 *     MultilinearPolynomial::evaluate.  The Fiat-Shamir transcript (Keccak256Transcript) stays on the caller's side:
 *     every round passes its message to `challenge` and receives the verifier's challenge.  Polynomials: 2^num_rounds elements,
 *     Montgomery form, index bit (num_rounds - 1) = the first variable (bound first), as in Arecibo's MultilinearPolynomial.
 *     Not here: the transcript, proof (de)serialisation, the verifiers (HyperKZG's pairing check) -- CPU / third-party protocol code.
 * ------------------------------------------------------------------------------------------------- */
/* message: the round's prover message in `fmt` -- sum-check: s(0) | s(1) | s(2) [| s(3)] (32 bytes each; Arecibo absorbs the
 * compressed form, i.e. the coefficients without the linear one: the caller converts);  IPA: L | R as 96-byte points.
 * Writes the challenge (32 bytes, `fmt`) and returns 0, or non-zero to abort the proof. */
typedef int (*lurk_challenge_fn)(void *user, int round, const uint8_t *message, size_t message_len, uint8_t challenge_out[32]);
#define LURK_SUMCHECK_QUAD 0  /* claim = sum_i A[i] B[i]                 d_polys = {A, B}          degree 2 */
#define LURK_SUMCHECK_CUBIC 1 /* claim = sum_i A[i] (B[i] C[i] - D[i])   d_polys = {A, B, C, D}    degree 3 */
/* Runs all num_rounds rounds.  The polynomials are consumed (bound in place; element 0 of each ends as its final evaluation).
 * round_evals: num_rounds x (degree + 1) x 32 bytes; challenges: num_rounds x 32; final_evals: 2 or 4 x 32 (any may be NULL). */
int lurk_sumcheck_prove_dev(int field_id, int kind, void *const *d_polys, int num_rounds, const uint8_t claim[32],
                            lurk_challenge_fn challenge, void *user, uint8_t *round_evals, uint8_t *challenges, uint8_t *final_evals,
                            int fmt, void *stream);
/* SumcheckProof::prove_quad_batch / prove_cubic_with_additive_term_batch (BatchedRelaxedR1CSSNARK: SuperNova's `compress`,
 * src/proof/supernova.rs:293-317): n_instances (<= 60) claims proven together, the round message is sum_i coeffs[i] * s_i(X).
 * Instance i has 2 or 4 polynomials of 2^num_rounds[i] elements (d_polys instance-major) and joins in round max - num_rounds[i];
 * before that its round polynomial is the constant 2^(remaining - num_rounds[i] - 1) * claims[i].  coeffs may be NULL (all 1).
 * round_evals: max_rounds x (degree + 1) x 32; challenges: max_rounds x 32; final_evals: n_instances x (2 | 4) x 32. */
int lurk_sumcheck_prove_batch_dev(int field_id, int kind, int n_instances, void *const *d_polys, const int *num_rounds,
                                  const uint8_t *claims, const uint8_t *coeffs, lurk_challenge_fn challenge, void *user,
                                  uint8_t *round_evals, uint8_t *challenges, uint8_t *final_evals, int fmt, void *stream);
/* EqPolynomial::new(tau).evals(): d_out[i] = prod_j (bit_j(i) ? tau[j] : 1 - tau[j]), tau[0] <-> the top index bit; 2^num_vars
 * elements in `fmt` (tau: host, num_vars x 32 bytes, same fmt). */
int lurk_eq_evals_dev(int field_id, const uint8_t *tau, int num_vars, void *d_out, int fmt, void *stream);
/* <a, b> over n Montgomery elements (MultilinearPolynomial::evaluate = <Z, eq(r)>; the c_L / c_R of an IPA round).  Synchronous. */
int lurk_inner_product_dev(int field_id, const void *d_a, const void *d_b, size_t n, uint8_t out[32], int fmt, void *stream);
/* PolyEvalWitness::batch_diff_size (batch_eval_reduce's joint polynomial): d_out[i] = sum_{j : i < lens[j]} coeffs[j] * P_j[i] for
 * i < out_len, zero where no P_j reaches -- every P_j zero-extended at the end.  n_polys <= 120 device polynomials of lens[j] <= out_len
 * Montgomery elements (d_polys / lens / coeffs: host arrays; coeffs: n_polys x 32 bytes in `fmt`).  d_out must not overlap any P_j.
 * One launch; asynchronous on `stream`. */
int lurk_poly_combine_dev(int field_id, int n_polys, const void *const *d_polys, const size_t *lens, const uint8_t *coeffs, void *d_out,
                          size_t out_len, int fmt, void *stream);
/* one IPA folding step, in place on the first n / 2 slots: a[i] <- x a[i] + y a[i + n/2];  G[i] <- x G[i] + y G[i + n/2]
 * (CommitmentKey::fold; bases affine Montgomery; x, y host scalars in `fmt`). */
int lurk_ipa_fold_scalars_dev(int field_id, void *d_a, size_t n, const uint8_t x[32], const uint8_t y[32], int fmt, void *stream);
int lurk_ipa_fold_bases_dev(int curve_id, void *d_bases_mont, size_t n, const uint8_t x[32], const uint8_t y[32], int fmt, void *stream);
/* All log_n rounds of InnerProductArgument::prove on device-resident a, b (2^log_n scalars each, Montgomery, consumed) under the
 * key of context `ck` (>= 2^log_n bases; NOT consumed): per round c_L = <a_lo, b_hi>, c_R = <a_hi, b_lo>,
 * L = commit(a_lo; G_hi) + c_L ck_c, R = commit(a_hi; G_lo) + c_R ck_c, r = challenge(L | R), a' = a_lo r + a_hi / r,
 * b' = b_lo / r + b_hi r, G' = G_lo / r + G_hi r.  The folded key G' is never materialised: the prover only needs commitments under
 * it, and those are Pippenger passes over the original key with scalars weighted by the products of the earlier challenges
 * (lurk_ipa_fold_bases_dev is the explicit CommitmentKey::fold for callers that want G').  ck_c: the (already scaled) base for the
 * inner-product value, 64 bytes affine in `fmt`.  L_out / R_out: log_n x 96 bytes. */
int lurk_ipa_prove_dev(int curve_id, lurk_msm_ctx *ck, const uint8_t ck_c[64], void *d_a, void *d_b, int log_n,
                       lurk_challenge_fn challenge, void *user, uint8_t *L_out, uint8_t *R_out, uint8_t a_final[32], uint8_t b_final[32],
                       int fmt, void *stream);
/* provider::hyperkzg::EvaluationEngine::prove (the opening argument of the primary BN256 circuit, EE1 in src/proof/nova.rs:65-71):
 * d_poly = 2^num_vars evaluations (Montgomery, not modified), point = num_vars elements (host, `fmt`), ck = a context on the KZG key
 * (>= 2^num_vars bases).  Phase 1: P_{i+1}[j] = P_i[2j] + x_{l-1-i} (P_i[2j+1] - P_i[2j]) and com_i = commit(P_i), i = 1..l-1;
 * challenge(round 0, com) -> r; u = (r, -r, r^2); v[t][j] = P_j(u_t); challenge(round 1, v) -> q; B = sum_j q^j P_j;
 * w_t = commit(B(X) / (X - u_t)); challenge(round 2, w) is called for the transcript's sake.
 * com_out: (num_vars - 1) x 96; w_out: 3 x 96; v_out: 3 x num_vars x 32 (v[t][j] at (t * num_vars + j)). */
int lurk_hyperkzg_prove_dev(int curve_id, lurk_msm_ctx *ck, const void *d_poly, const uint8_t *point, int num_vars,
                            lurk_challenge_fn challenge, void *user, uint8_t *com_out, uint8_t *w_out, uint8_t *v_out, int fmt,
                            void *stream);

/* ---------------------------------------------------------------------------------------------------
 * S5  Fold helpers on device-resident vectors (Arecibo NIFS::prove / R1CSShape::commit_T /
 *     RelaxedR1CSWitness::fold; SURVEY.md Appendix B).  All vectors Montgomery form on the device.
 * ------------------------------------------------------------------------------------------------- */
/* out[i] = a[i] + r * b[i]  (W <- W1 + r W2, E <- E1 + r T).  r: 32 bytes host, Montgomery. out may alias a. */
int lurk_axpy_dev(int field_id, const void *d_a, const void *d_b, const uint8_t r_mont[32], size_t n, void *d_out,
                  void *stream);
/* y = M z for a CSR matrix (row_ptr: rows+1 x u64, col: nnz x u32, val: nnz elements) */
int lurk_spmv_csr_dev(int field_id, const void *d_row_ptr, const void *d_col, const void *d_val, size_t rows,
                      const void *d_z, void *d_y, void *stream);
/* T = az1*bz2 + az2*bz1 - u1*cz2 - u2*cz1 */
int lurk_cross_term_dev(int field_id, const void *d_az1, const void *d_bz1, const void *d_cz1, const void *d_az2,
                        const void *d_bz2, const void *d_cz2, const uint8_t u1_mont[32], const uint8_t u2_mont[32],
                        size_t n, void *d_t, void *stream);
/* element-wise format conversion on the device (LURK_FMT_*), in place allowed */
int lurk_convert_dev(int field_id, const void *d_in, size_t n, int to_fmt, void *d_out, void *stream);

/* ---------------------------------------------------------------------------------------------------
 * S5/S6  Fold context: the GPU half of `Proof::prove_recursively` (src/proof/nova.rs:260-339, supernova.rs:207-291) for
 *     ONE running instance, i.e. what RecursiveSNARK::new / prove_step (nova.rs:286-293) do with the primary circuit's
 *     witness inside Arecibo's NIFS::prove (SURVEY.md Appendix B), on device-resident state:
 *         comm_W2 = commit(W2); T = cross term; comm_T = commit(T); r = RO(..., comm_W2, ..., comm_T);
 *         (W, u, X) += r (W2, 1, X2); E += r T; comm_W += r comm_W2; comm_E += r comm_T.
 *     The reference overlaps a witness thread with the fold thread over a bounded channel (nova.rs:297-326); here stage A
 *     (inputs, slot witnesses, commit(W2), A z2 .. C z2) of up to `depth - 1` later steps runs on its own CUDA streams while
 *     stage B -- the sequential chain -- runs without any host round trip: the commitments are finished, exchanged between
 *     GPUs (peer memory over NVLink), normalised, hashed into the challenge and consumed by the fold on the device.
 *     SuperNova / NIVC: one context per circuit index (src/lem/multiframe.rs:941), all sharing one commitment key.
 *     z = (W, u, X).  Matrices are CSR over z's columns.  All calls of one context must come from one thread at a time.
 * ------------------------------------------------------------------------------------------------- */
typedef struct lurk_fold_ctx lurk_fold_ctx;
typedef struct lurk_fold_config {
    int curve_id;            /* commitments on this curve; the witness field is its scalar field */
    int depth;               /* fresh-instance buffers, 1..4: stage A may run depth - 1 steps ahead of the fold */
    uint64_t n_w;            /* |W| of this rank's share */
    uint64_t n_x;            /* |X| (2 for Nova step circuits) */
    uint64_t n_rows;         /* constraints of this rank's share */
    const uint64_t *row_ptr[3]; /* A, B, C: rows + 1 offsets                                    (host) */
    const uint32_t *col[3];     /* column of every non-zero, < n_w + 1 + n_x                     (host) */
    const uint8_t *val[3];      /* coefficient of every non-zero, 32 bytes each, in `fmt`        (host) */
    int fmt;
    int world, rank;         /* > 1: the key is sharded; the partial commitments are exchanged every step */
    int latency_sms;         /* 0 = off; otherwise SMs reserved for the latency-shaped kernels of the chain (green
                                contexts; multiple of 8, e.g. 16): bucket accumulation and stage A get the rest */
} lurk_fold_config;
/* ck_w / ck_t: this rank's bases for W (>= n_w points) and for T / E (>= n_rows points); the same context when the key is
 * not sharded.  Fixed-base tables are built if absent.  The contexts must outlive the fold context. */
int lurk_fold_ctx_create(const lurk_fold_config *cfg, lurk_msm_ctx *ck_w, lurk_msm_ctx *ck_t, lurk_fold_ctx **out);
void lurk_fold_ctx_destroy(lurk_fold_ctx *ctx);
/* One batch per slot type of the step circuit (generate_slots_witnesses, src/lem/multiframe.rs:520-592): arity 3/4/6/8 =
 * Poseidon slots, 0 = bit-decomposition slots.  offsets[k] = element offset of block k inside W (the reference's layout:
 * every frame's aux = [its slot blocks | LEM body aux], multiframe.rs:635-712).  Returns the batch index (>= 0). */
int lurk_fold_ctx_add_slot_batch(lurk_fold_ctx *ctx, int arity, size_t count, const uint64_t *offsets);
/* The parts of W2 the host produces (LEM body aux, the augmented-circuit part): up to 4 strided spans of W; the host
 * buffer LURK_FOLD_BUF_GLUE holds them densely, span after span, row after row. */
typedef struct lurk_fold_span { uint64_t first, row_elems, stride, rows; } lurk_fold_span;
int lurk_fold_ctx_set_spans(lurk_fold_ctx *ctx, int n_spans, const lurk_fold_span *spans);
/* Random oracle = Arecibo's PoseidonRO (neptune sponge, arity 24, [Absorb(n), Squeeze(1)], low `challenge_bits` bits).
 * kinds[i] says what is absorbed at position i.  Default (NIFS::prove): CONST pp_digest, W_X, W_Y, W_INF, CONST X2[0],
 * CONST X2[1], T_X, T_Y, T_INF with 128 bits.  CONST values come from the host buffer LURK_FOLD_BUF_RO of the step. */
#define LURK_FOLD_RO_CONST 0
#define LURK_FOLD_RO_W_X 1
#define LURK_FOLD_RO_W_Y 2
#define LURK_FOLD_RO_W_INF 3
#define LURK_FOLD_RO_T_X 4
#define LURK_FOLD_RO_T_Y 5
#define LURK_FOLD_RO_T_INF 6
int lurk_fold_ctx_set_ro(lurk_fold_ctx *ctx, int n_absorb, const int *kinds, int challenge_bits);
/* Pinned host buffers the caller (the CPU witness generator) fills before stage A of buffer b: `which` >= 0 = preimages
 * of that slot batch (count * arity elements; bit decomposition: count values), or one of the names below. */
#define LURK_FOLD_BUF_GLUE (-1) /* the spans, densely                       (witness field)            */
#define LURK_FOLD_BUF_X2 (-2)   /* public IO of the fresh instance, n_x      (witness field)            */
#define LURK_FOLD_BUF_RO (-3)   /* 24 elements: position i = CONST value of RO slot i (commitment curve's base field) */
#define LURK_FOLD_BUF_W2 (-4)   /* device only: z2 of buffer b = (W2, 1, X2), Montgomery               */
#define LURK_FOLD_BUF_T (-5)    /* device only: cross term of the last step                             */
#define LURK_FOLD_BUF_Z1 (-6)   /* device only: running z = (W, u, X)                                   */
#define LURK_FOLD_BUF_E1 (-7)   /* device only: running E                                               */
int lurk_fold_ctx_host_buffer(lurk_fold_ctx *ctx, int b, int which, void **ptr, size_t *bytes);
int lurk_fold_ctx_device_buffer(lurk_fold_ctx *ctx, int b, int which, void **d_ptr, size_t *bytes);
/* Sharded key, one process per GPU: every rank publishes a 64-byte handle of its exchange buffer (any transport: e.g. a
 * torch.distributed all_gather of the bytes) and receives all `world` handles, ordered by rank. */
int lurk_fold_ctx_exchange_handle(lurk_fold_ctx *ctx, uint8_t handle[64]);
int lurk_fold_ctx_set_peers(lurk_fold_ctx *ctx, const uint8_t *handles /* world * 64 bytes */);
/* Running instance (checkpoint / resume: prove_recursively's `init: Option<RecursiveSNARK>`, src/proof/mod.rs:107-115).
 * comm_* are 96-byte points x | y | z as everywhere in this header; any output pointer of _get_ may be NULL. */
int lurk_fold_ctx_set_running(lurk_fold_ctx *ctx, const uint8_t *W, const uint8_t *E, const uint8_t u[32], const uint8_t *X,
                              const uint8_t comm_W[96], const uint8_t comm_E[96], int fmt);
int lurk_fold_ctx_get_running(lurk_fold_ctx *ctx, uint8_t *W, uint8_t *E, uint8_t u[32], uint8_t *X, uint8_t comm_W[96],
                              uint8_t comm_E[96], int fmt);
/* Stage A of the step whose inputs are in the host buffers of b (fmt = their format).  LURK_FOLD_INPUTS_RESIDENT: skip
 * the host-to-device copies and use what the device buffers hold (Montgomery). Asynchronous. */
#define LURK_FOLD_INPUTS_RESIDENT 1
int lurk_fold_ctx_stage_a(lurk_fold_ctx *ctx, int b, int flags, int fmt);
/* RecursiveSNARK::new: the running instance becomes the fresh instance of buffer b (u = 1, E = 0, comm_E = identity). */
int lurk_fold_ctx_init_running(lurk_fold_ctx *ctx, int b);
/* Stage B: enqueues the whole fold of the fresh instance in buffer b onto the running instance.  Asynchronous; call
 * stage_a for later steps and stage_b_launch for the next step without waiting. */
int lurk_fold_ctx_stage_b_launch(lurk_fold_ctx *ctx, int b);
typedef struct lurk_fold_result {
    uint8_t comm_W[96];         /* commitment to the fresh witness (whole key) */
    uint8_t comm_T[96];         /* commitment to the cross term; identity after init_running */
    uint8_t r[32];              /* the challenge as an element of the witness field */
    uint8_t running_comm_W[96]; /* after this step's fold */
    uint8_t running_comm_E[96];
    uint8_t ro_hash[32];        /* the squeezed sponge element before truncation (commitment curve's base field) */
    int status;
    uint64_t seq;               /* exchange epoch = number of commitments finished by this context */
} lurk_fold_result;
/* waits for the step enqueued on buffer b (init_running or stage_b_launch) and returns its record */
int lurk_fold_ctx_collect(lurk_fold_ctx *ctx, int b, lurk_fold_result *out, int fmt);
/* Verifier-side sanity of the running instance, computed on the device: rows with (A z) o (B z) != u (C z) + E, and
 * whether commit(W) / commit(E) recomputed from the vectors equal the folded commitments.  Synchronous. */
int lurk_fold_ctx_check_running(lurk_fold_ctx *ctx, uint64_t *bad_rows, int *comm_W_ok, int *comm_E_ok);
/* kernels enqueued by the last stage A / stage B, device time of the bucket-accumulation kernels of the last commit(W2) of
 * buffer 0 and of the last commit(T) (CUDA events on the launching streams).  Synchronises the context. */
int lurk_fold_ctx_stats(lurk_fold_ctx *ctx, unsigned *launches_a, unsigned *launches_b, float *accumulate_w_ms, float *accumulate_t_ms);
int lurk_fold_ctx_sync(lurk_fold_ctx *ctx);

/* ---------------------------------------------------------------------------------------------------
 * K6  Number-theoretic transform (north_star; no call site in the reference -- SURVEY.md D4).
 *     In-place length-2^log_n DFT over the field's 2-adic subgroup, natural order in and out, Montgomery form.
 *     Roots: omega = g^((p-1)/2^s) with g the multiplicative generator of halo2curves / pasta_curves.
 * ------------------------------------------------------------------------------------------------- */
int lurk_ntt_dev(int field_id, void *d_data, int log_n, int inverse, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* LURK_B200_H */
