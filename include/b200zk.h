/* libb200zk -- C ABI of the B200-native Groth16 (BLS12-381) proving backend.
 *
 * This is the drop-in boundary for the prove path of ArielElb/zkSnark-FinalProject.
 * The reference has no FFI of its own: its handlers call the arkworks trait
 * surface directly, so each entry point below names the arkworks call (and the
 * reference call site) it replaces.  A Rust shim (INTEGRATION.md) packs arkworks
 * values into these plain buffers; nothing here mentions torch or C++ types.
 *
 * Data layouts (identical to arkworks' in-memory forms, so the shim copies limbs):
 *   Fr element   : 4 x uint64 little-endian limbs, Montgomery form, R = 2^256
 *                  (ark_ff::Fp<MontBackend<FrConfig,4>,4>.0.0)
 *   Fr "bigint"  : 4 x uint64 little-endian limbs, canonical (into_bigint())
 *   Fq element   : 6 x uint64 limbs, Montgomery form, R = 2^384
 *   G1 affine    : x, y            -> 12 x uint64 (96 B); infinity flagged separately
 *   G2 affine    : x.c0, x.c1, y.c0, y.c1 -> 24 x uint64 (192 B)
 *   infinity map : 1 bit per point, bit i of byte i/8 (LSB first); NULL = no
 *                  point is the identity
 *   projective   : X, Y, Z Jacobian as arkworks' Projective {x, y, z}; Z = 0 is
 *                  the identity
 *
 * Threading: a b2z_ctx serialises the calls made on it (internal mutex); use one
 * ctx per host thread (actix worker, /root/reference/src/main.rs:37) for
 * concurrency.  A b2z_pk / b2z_r1cs handle holds per-proof device scratch and
 * therefore BELONGS TO THE CONTEXT IT WAS UPLOADED THROUGH: passing it to any
 * other context returns B2Z_EINVAL (upload one copy per context / worker).
 * Errors never unwind across the boundary: every call returns a b2z_status and
 * b2z_last_error() describes the most recent failure on that ctx.
 *
 * Assignment pointers (`z`) of the *_r1cs and shard entry points may be host
 * pointers (pageable or page-locked) or device pointers on the context's device
 * (the copy uses cudaMemcpyDefault); a device buffer must be complete when the
 * call is made.
 */
#ifndef B200ZK_H_
#define B200ZK_H_

#include <stddef.h>
#include <stdint.h>

#if defined(__GNUC__)
#define B2Z_API __attribute__((visibility("default")))
#else
#define B2Z_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

typedef int32_t b2z_status;
enum {
  B2Z_OK = 0,
  B2Z_EINVAL = 1,  /* bad argument (NULL buffer, inconsistent sizes)                */
  B2Z_ESIZE = 2,   /* domain too large: log_n > 32 (ark-poly returns None ->
                      SynthesisError::PolynomialDegreeTooLarge)                     */
  B2Z_ECUDA = 3,   /* CUDA runtime failure, incl. "no CUDA device": there is no
                      CPU fallback                                                  */
  B2Z_ENOMEM = 4   /* device or pinned-host allocation failed                       */
};

typedef struct b2z_ctx b2z_ctx;
typedef struct b2z_pk b2z_pk;

/* One context per (host thread, device).  device_id is a CUDA ordinal. */
B2Z_API b2z_status b2z_ctx_create(int device_id, b2z_ctx** out);
B2Z_API void b2z_ctx_destroy(b2z_ctx* ctx);
B2Z_API const char* b2z_last_error(const b2z_ctx* ctx);

/* ---- ark_poly::Radix2EvaluationDomain<Fr> -------------------------------------
 * Replaces fft_in_place / ifft_in_place on `domain` and on
 * `domain.get_coset(g)` (used by LibsnarkReduction::witness_map_from_matrices,
 * reached from Groth16::prove at src/arkworks/backend/matrix_proof.rs:139).
 * data: n = 2^log_n Fr elements (host memory), transformed in place, natural
 * order in and out.  coset_gen: NULL for the base domain, else the coset offset
 * g as an Fr element; forward evaluates at g*w^k, inverse undoes exactly that. */
B2Z_API b2z_status b2z_ntt_fr(b2z_ctx* ctx, uint64_t* data, uint32_t log_n, int inverse,
                      const uint64_t coset_gen[4]);

/* ---- ark_groth16::r1cs_to_qap::LibsnarkReduction::witness_map_from_matrices ----
 * after its sparse row evaluations: a, b, c are the length-n (n = 2^log_n)
 * evaluation vectors (a[num_constraints + j] = z[j] already placed, zero padded);
 * h_out receives the n coefficients of (A*B - C)/Z_H, natural order.             */
B2Z_API b2z_status b2z_witness_map(b2z_ctx* ctx, const uint64_t* a, const uint64_t* b,
                           const uint64_t* c, uint32_t log_n, uint64_t* h_out);

/* ---- ark_ec::VariableBaseMSM::msm_bigint --------------------------------------
 * for G1Projective / G2Projective (called five times per proof by
 * create_proof_with_assignment).  bases: n affine points; scalars: n canonical
 * bigints < 2^255 (into_bigint() of an Fr element; anything larger is rejected
 * with B2Z_EINVAL); out: one Jacobian point (18 / 36 limbs), canonical Montgomery
 * limbs.                                                                          */
B2Z_API b2z_status b2z_msm_g1(b2z_ctx* ctx, const uint64_t* bases, const uint8_t* inf_bitmap,
                      const uint64_t* scalars, uint64_t n, uint64_t out_xyz[18]);
B2Z_API b2z_status b2z_msm_g2(b2z_ctx* ctx, const uint64_t* bases, const uint8_t* inf_bitmap,
                      const uint64_t* scalars, uint64_t n, uint64_t out_xyz[36]);

/* ---- ark_groth16::ProvingKey<Bls12_381> ---------------------------------------
 * Uploaded once per circuit (the reference re-runs setup per request,
 * matrix_proof.rs:129; a shim may cache by circuit shape), then proved against
 * many times.  All arrays are copied; the caller keeps ownership.               */
typedef struct b2z_pk_desc {
  uint64_t num_variables;    /* m: instance (incl. the constant 1) + witness              */
  uint64_t num_instance;     /* l                                                          */
  uint32_t log_domain;       /* n = 2^log_domain                                           */
  const uint64_t* a_query;   const uint8_t* a_inf;      /* m  G1 */
  const uint64_t* b_g1_query; const uint8_t* b_g1_inf;  /* m  G1 */
  const uint64_t* b_g2_query; const uint8_t* b_g2_inf;  /* m  G2 */
  const uint64_t* h_query;   const uint8_t* h_inf;      /* n - 1  G1 */
  const uint64_t* l_query;   const uint8_t* l_inf;      /* m - l  G1 */
  const uint64_t* alpha_g1;  /* vk.alpha_g1  (12 limbs) */
  const uint64_t* beta_g1;   /* pk.beta_g1               */
  const uint64_t* delta_g1;  /* pk.delta_g1              */
  const uint64_t* beta_g2;   /* vk.beta_g2   (24 limbs) */
  const uint64_t* delta_g2;  /* vk.delta_g2              */
} b2z_pk_desc;

B2Z_API b2z_status b2z_pk_upload(b2z_ctx* ctx, const b2z_pk_desc* desc, b2z_pk** out);
B2Z_API void b2z_pk_free(b2z_ctx* ctx, b2z_pk* pk);

/* ---- ark_groth16::Groth16::<Bls12_381>::create_proof_with_reduction ------------
 * minus circuit synthesis (which stays in Rust): the call at
 * fibbonaci_handler.rs:110, matrix_proof.rs:139-140, prime_snark.rs:119.
 *   a/b/c_evals : as for b2z_witness_map (n = 2^pk.log_domain elements each)
 *   z           : full assignment, m Fr elements (Montgomery), z[0] = 1
 *   r, s        : the prover's two Fr::rand draws (Montgomery), made by the host
 *   proof_out   : Proof::serialize_compressed bytes, A(48) | B(96) | C(48)
 *                 (what encode_proof base64-encodes, matrix_proof_of_work/io.rs:48) */
B2Z_API b2z_status b2z_groth16_prove(b2z_ctx* ctx, const b2z_pk* pk, const uint64_t* a_evals,
                             const uint64_t* b_evals, const uint64_t* c_evals,
                             const uint64_t* z, const uint64_t r[4], const uint64_t s[4],
                             uint8_t proof_out[192]);

/* ---- constraint matrices on the device (ark_relations ConstraintMatrices) ---------------------
 * The `evaluate_constraint` loop of LibsnarkReduction::witness_map_from_matrices: upload the three
 * R1CS matrices once per circuit as CSR (row_ptr: num_constraints + 1 offsets; cols: variable
 * indices into z = instance || witness; coeffs: Fr Montgomery limbs, 4 per entry), then each proof
 * sends only the assignment z.  b2z_witness_map_from_matrices is the whole arkworks function;
 * b2z_groth16_prove_r1cs is b2z_groth16_prove with the row evaluation done on the GPU.          */
typedef struct b2z_r1cs b2z_r1cs;
B2Z_API b2z_status b2z_r1cs_upload(b2z_ctx* ctx, uint64_t num_constraints, uint64_t num_instance,
                                   uint64_t num_variables,
                                   const uint64_t* a_row_ptr, const uint32_t* a_cols, const uint64_t* a_coeffs,
                                   const uint64_t* b_row_ptr, const uint32_t* b_cols, const uint64_t* b_coeffs,
                                   const uint64_t* c_row_ptr, const uint32_t* c_cols, const uint64_t* c_coeffs,
                                   b2z_r1cs** out);
B2Z_API void b2z_r1cs_free(b2z_ctx* ctx, b2z_r1cs* r1cs);
B2Z_API b2z_status b2z_r1cs_eval(b2z_ctx* ctx, b2z_r1cs* r1cs, const uint64_t* z, uint64_t* a_out, uint64_t* b_out,
                                 uint64_t* c_out);
/* y = M x over Fr for a one-off CSR matrix (host buffers; x, coeffs, y Montgomery limbs).  Key
 * generation uses it for the QAP evaluation at tau (the transposed matrices times the Lagrange
 * coefficients: LibsnarkReduction::instance_map_with_evaluation).                                */
B2Z_API b2z_status b2z_spmv_fr(b2z_ctx* ctx, uint64_t nrows, uint64_t ncols, const uint64_t* row_ptr,
                               const uint32_t* cols, const uint64_t* coeffs, const uint64_t* x, uint64_t* y_out);
B2Z_API b2z_status b2z_witness_map_from_matrices(b2z_ctx* ctx, b2z_r1cs* r1cs, const uint64_t* z, uint64_t* h_out);
B2Z_API b2z_status b2z_groth16_prove_r1cs(b2z_ctx* ctx, const b2z_pk* pk, b2z_r1cs* r1cs, const uint64_t* z,
                                          const uint64_t r[4], const uint64_t s[4], uint8_t proof_out[192]);

/* ---- point-sharded proving across the GPUs of one box ------------------------------------
 * An MSM is a sum over independent (scalar, point) pairs, so a proof shards by points
 * (SURVEY.md 8(e)): rank k of `world` keeps, of the a / b_g1 / b_g2 / l queries, the variables of
 * blocks k, k + world, k + 2 world, ... (blocks of 64 variables: Groth16 assignments have long stretches
 * of small / Boolean values, and contiguous ranges left some GPUs with a third of the others' work), and
 * the contiguous chunk [n k/world, n (k+1)/world) of the (bit-reversed) h bases; rank 0 also
 * keeps the alpha/beta/delta terms.  Every rank passes the SAME full desc and the same full
 * a/b/c/z/r/s; the witness map runs on every rank.  Each rank gets B2Z_PARTIAL_BYTES of partial
 * sums (XYZZ limbs: A | s*A | r*B1 | L | H in G1, B in G2 -- scalar multiplication is linear, so
 * every rank applies s and r to its own partial A and B1); gather them over any transport (NCCL
 * all_gather of 1344 bytes per rank) and finish on the host with b2z_groth16_combine.         */
#define B2Z_PARTIAL_BYTES 1344
B2Z_API b2z_status b2z_pk_upload_shard(b2z_ctx* ctx, const b2z_pk_desc* desc, uint32_t rank, uint32_t world,
                                       b2z_pk** out);
/* The same with an explicit slice: variables / h positions [total * from / den, total * to / den); the slice with
 * from == 0 keeps the alpha/beta/delta terms.  Lets a caller give lighter shards to the GPUs that also transform one
 * of the witness-map inputs (b2z_r1cs_coset_evals).  The slices of a proof must tile [0, den) in rank order.     */
B2Z_API b2z_status b2z_pk_upload_slice(b2z_ctx* ctx, const b2z_pk_desc* desc, uint32_t from, uint32_t to, uint32_t den,
                                       b2z_pk** out);
B2Z_API b2z_status b2z_groth16_prove_partial(b2z_ctx* ctx, const b2z_pk* pk, const uint64_t* a_evals,
                                             const uint64_t* b_evals, const uint64_t* c_evals, const uint64_t* z,
                                             const uint64_t r[4], const uint64_t s[4], uint8_t* partial_out);
/* the same with the constraint rows evaluated on the GPU: only z crosses PCIe on every rank */
B2Z_API b2z_status b2z_groth16_prove_partial_r1cs(b2z_ctx* ctx, const b2z_pk* pk, b2z_r1cs* r1cs, const uint64_t* z,
                                                  const uint64_t r[4], const uint64_t s[4], uint8_t* partial_out);
/* host only (no GPU, no ctx): partials = world x B2Z_PARTIAL_BYTES in rank order */
B2Z_API b2z_status b2z_groth16_combine(const uint8_t* partials, uint32_t world, uint8_t proof_out[192]);

/* Same computation on inputs already resident in device memory (device pointers
 * on ctx's device; a/b/c are clobbered).  The buffers must be complete, or have
 * been produced on the legacy default stream (the library orders its own streams
 * after that stream; it does not synchronise the device).  The proof bytes still
 * land in host memory.                                                           */
B2Z_API b2z_status b2z_groth16_prove_device(b2z_ctx* ctx, const b2z_pk* pk, uint64_t* d_a,
                                    uint64_t* d_b, uint64_t* d_c, const uint64_t* d_z,
                                    const uint64_t r[4], const uint64_t s[4],
                                    uint8_t proof_out[192]);

/* ---- ark_ec::scalar_mul::fixed_base::FixedBase::msm ------------------------------
 * on the standard generators: out[i] = scalars[i] * G.  ark-groth16's setup builds
 * every query array this way (Groth16::setup, matrix_proof.rs:129); the benchmarks
 * use it to make synthetic bases.  scalars: canonical bigints; out: affine points
 * (12 / 24 limbs each); out_inf: identity bitmap, (n + 7) / 8 bytes.                */
B2Z_API b2z_status b2z_fixed_base_mul_g1(b2z_ctx* ctx, const uint64_t* scalars, uint64_t n,
                                         uint64_t* out_points, uint8_t* out_inf);
B2Z_API b2z_status b2z_fixed_base_mul_g2(b2z_ctx* ctx, const uint64_t* scalars, uint64_t n,
                                         uint64_t* out_points, uint8_t* out_inf);

/* ---- ark_groth16::generator::generate_parameters_with_qap::<LibsnarkReduction> on the device --------------------
 * Groth16::setup (matrix_proof.rs:128-131, fibbonaci_handler.rs:107, prime_snark.rs:111-115) after its random draws:
 * the caller passes the toxic waste and the generators (ark draws alpha, beta, gamma, delta, then g1, g2, then tau).
 * The matrices are those of b2z_r1cs_upload (same context).  Lagrange coefficients at tau, the QAP evaluation, the
 * scalars and every fixed-base multiplication run on the GPU; the key is assembled in device memory and returned
 * as a handle equal to what b2z_pk_upload makes from the same arrays (ready for b2z_groth16_prove / _prove_r1cs).
 * Every input is checked on the host before any GPU work; B2Z_EINVAL with a message for: an element >= r, gamma or
 * delta = 0, tau in the domain (tau^n = 1), a generator that is the identity, off the curve or outside the r-order
 * subgroup, an r1cs of another context.  Size limits: those of b2z_pk_upload.                                     */
typedef struct b2z_setup_desc {
  const uint64_t* alpha; const uint64_t* beta; const uint64_t* gamma; const uint64_t* delta; const uint64_t* tau;
                                   /* Fr, Montgomery limbs, each < r; gamma, delta != 0; tau^n != 1 */
  const uint64_t* g1_generator;    /* affine, 12 limbs; NULL = the standard generator */
  const uint64_t* g2_generator;    /* affine, 24 limbs; NULL = the standard generator */
} b2z_setup_desc;
typedef struct b2z_vk_out {        /* filled by the call */
  uint64_t alpha_g1[12], beta_g2[24], gamma_g2[24], delta_g2[24];
  uint64_t* gamma_abc_g1;          /* caller-allocated, num_instance x 12 */
  uint8_t*  gamma_abc_inf;         /* caller-allocated, (num_instance + 7) / 8 */
} b2z_vk_out;
B2Z_API b2z_status b2z_groth16_setup(b2z_ctx* ctx, b2z_r1cs* r1cs, const b2z_setup_desc* desc,
                                     b2z_pk** pk_out, b2z_vk_out* vk_out);
/* The same setup straight into shard `rank` of `world`: each rank does only its own shard's fixed-base
 * multiplications and window copies, and no query point leaves device memory.  Every rank passes the same desc
 * and the same matrices (uploaded through its own context).
 *  - *pk_out equals what b2z_pk_upload_shard(rank, world) makes from the arrays that b2z_pk_download returns for
 *    b2z_groth16_setup's key, for the same desc and matrices.  Same sharding rule: variables in blocks of 64,
 *    block-cyclic over the ranks; contiguous ranges instead when num_instance > 64; h positions in the contiguous
 *    chunk [n rank/world, n (rank+1)/world) of the bit-reversed order; the alpha/beta/delta terms on rank 0 only;
 *    precomputed window copies when 1/world of a whole key's copies fit in half the free device memory, decided
 *    before the call's own allocations.  The shard is ready for b2z_groth16_prove_partial[_r1cs],
 *    b2z_groth16_shard_* and b2z_dist_create.
 *  - vk_out holds the full verifying key on every rank, identical across ranks.
 *  - world == 1 gives the whole key: downloadable, and byte-equal to b2z_groth16_setup's key.
 *  - rank >= world or world == 0: B2Z_EINVAL and *pk_out = NULL.  All of b2z_groth16_setup's checks apply unchanged
 *    and run on the host before any GPU work.  b2z_pk_download on a shard returns B2Z_EINVAL.                     */
B2Z_API b2z_status b2z_groth16_setup_shard(b2z_ctx* ctx, b2z_r1cs* r1cs, const b2z_setup_desc* desc, uint32_t rank,
                                           uint32_t world, b2z_pk** pk_out, b2z_vk_out* vk_out);
/* A whole key (b2z_pk_upload or b2z_groth16_setup) back in the b2z_pk_desc layout: h_query in natural order, n - 1
 * points.  The arrays are caller-allocated with b2z_pk_desc's sizes (h: NULL when n = 1, l: NULL when m = l); the
 * counts and the five single points are filled by the call.  A shard returns B2Z_EINVAL.  For callers that persist a
 * key, or shard one with b2z_pk_upload_shard.                                                                       */
typedef struct b2z_pk_arrays {
  uint64_t num_variables;
  uint64_t num_instance;
  uint32_t log_domain;
  uint64_t* a_query;   uint8_t* a_inf;
  uint64_t* b_g1_query; uint8_t* b_g1_inf;
  uint64_t* b_g2_query; uint8_t* b_g2_inf;
  uint64_t* h_query;   uint8_t* h_inf;
  uint64_t* l_query;   uint8_t* l_inf;
  uint64_t alpha_g1[12], beta_g1[12], delta_g1[12], beta_g2[24], delta_g2[24];
} b2z_pk_arrays;
B2Z_API b2z_status b2z_pk_download(b2z_ctx* ctx, const b2z_pk* pk, b2z_pk_arrays* out);

/* ---- ark_groth16 verifier over the reference's wire formats (host only: no GPU, no ctx) -----------------
 * b2z_groth16_prepare_verifying_key = ark_groth16::prepare_verifying_key followed by
 * PreparedVerifyingKey::serialize_compressed -- the bytes encode_pvk base64-encodes
 * (src/arkworks/matrix_proof_of_work/io.rs:62-68; built at src/arkworks/backend/matrix_proof.rs:134-136):
 *   vk (alpha_g1 48 | beta_g2 96 | gamma_g2 96 | delta_g2 96 | u64 count | count x 48 gamma_abc_g1)
 *   | alpha_g1_beta_g2 (Fq12, 12 x 48 B little-endian) | gamma_g2_neg_pc | delta_g2_neg_pc
 *   (G2Prepared: u64 count | count x 3 x 96 B line coefficients | 1 B infinity flag).
 * Call with pvk_out == NULL to get the size in *pvk_len (40 106 + 48 num_instance bytes).
 * b2z_groth16_verify_with_processed_vk = Groth16::verify_with_processed_vk (matrix_proof.rs:199-206) on
 * those bytes, the 192 proof bytes and the public inputs (Fr Montgomery limbs, WITHOUT the leading 1):
 * *valid = 1 / 0; B2Z_EINVAL for malformed encodings or a wrong input count
 * (SynthesisError::MalformedVerifyingKey / a deserialization error in arkworks).                         */
typedef struct b2z_vk_desc {
  uint64_t num_instance;         /* length of gamma_abc_g1 (public inputs + 1)          */
  const uint64_t* alpha_g1;      /* 12 limbs                                            */
  const uint64_t* beta_g2;       /* 24 limbs                                            */
  const uint64_t* gamma_g2;
  const uint64_t* delta_g2;
  const uint64_t* gamma_abc_g1;  /* num_instance x 12 limbs                             */
  const uint8_t* gamma_abc_inf;  /* identity bitmap or NULL                             */
} b2z_vk_desc;
B2Z_API b2z_status b2z_groth16_prepare_verifying_key(const b2z_vk_desc* vk, uint8_t* pvk_out, uint64_t capacity,
                                                     uint64_t* pvk_len);
B2Z_API b2z_status b2z_groth16_verify_with_processed_vk(const uint8_t* pvk, uint64_t pvk_len,
                                                        const uint64_t* public_inputs, uint64_t num_inputs,
                                                        const uint8_t proof[192], int32_t* valid);

/* Groth16::verify_with_processed_vk for `count` proofs against ONE prepared verifying key, on ctx's GPU.
 *   pvk, pvk_len  : PreparedVerifyingKey::serialize_compressed bytes (as for b2z_groth16_verify_with_processed_vk)
 *   public_inputs : count x num_inputs Fr elements (Montgomery limbs, WITHOUT the leading 1), proof-major
 *   proofs        : count x 192 bytes (A 48 | B 96 | C 48, compressed)
 *   results       : count int32: 1 valid, 0 not valid, -1 = b2z_groth16_verify_with_processed_vk would return
 *                   B2Z_EINVAL for this proof alone (malformed encoding, point off the curve or outside the
 *                   subgroup, an input >= r)
 * For every i, results[i] is what b2z_groth16_verify_with_processed_vk gives for (pvk, inputs_i, proof_i): one
 * verdict per proof, not a single check of the whole batch.
 * B2Z_EINVAL, results not written: malformed pvk, num_inputs + 1 != the pvk's gamma_abc count, NULL buffers with
 * count > 0, a prepared G2 line list that is neither infinite nor 68 long (the host verifier's call-level errors).
 * B2Z_ESIZE: num_inputs > 1024.  count == 0: B2Z_OK, no GPU work.  Host buffers; proofs go through the device in
 * chunks of 65536, so device memory stays bounded whatever count is.                                              */
B2Z_API b2z_status b2z_groth16_verify_batch(b2z_ctx* ctx, const uint8_t* pvk, uint64_t pvk_len,
                                            const uint64_t* public_inputs, uint64_t num_inputs,
                                            const uint8_t* proofs, uint64_t count, int32_t* results);

/* ---- key-generation scalars on the host, multithreaded (row f3; no GPU, no ctx) ---------------------------------
 * ark_groth16's generate_parameters_with_qap (Groth16::setup, matrix_proof.rs:128-131) = O(n) scalar preparation + fixed-
 * base multiplications.  The multiplications are b2z_fixed_base_mul_g1/g2 (and b2z_spmv_fr for the QAP evaluation at
 * tau) on the GPU; these are the scalar part: exact element-wise vector operations over Fr, split over host threads
 * (threads = 0: all).  Elements are 4 x u64 Montgomery limbs; scalars (tau, base, scale, a, b, c) must be canonical (< r),
 * else B2Z_EINVAL; vector elements are reduced on load; outputs are canonical; `out` may alias an input.
 *   b2z_fr_lagrange_at   out[i] = L_i(tau) = Z(tau)/n * w^i / (tau - w^i), i < count <= n = 2^log_n, w the domain's
 *                        generator (LibsnarkReduction::instance_map_with_evaluation's evaluate_all_lagrange_coefficients);
 *                        B2Z_EINVAL when tau lies in the domain
 *   b2z_fr_geometric     out[i] = scale * base^i  (the h query's  tau^i Z(tau) / delta)
 *   b2z_fr_lincomb3      out[i] = a x[i] + b y[i] + c z[i]; a NULL vector drops its term  (beta A_i + alpha B_i + C_i, and
 *                        the gamma^-1 / delta^-1 scalings)
 *   b2z_fr_into_bigint   Montgomery -> canonical integer limbs (what b2z_fixed_base_mul_* and b2z_msm_* take)          */
B2Z_API b2z_status b2z_fr_lagrange_at(uint32_t log_n, const uint64_t tau[4], uint64_t count, uint32_t threads,
                                      uint64_t* out);
B2Z_API b2z_status b2z_fr_geometric(const uint64_t base[4], const uint64_t scale[4], uint64_t count, uint32_t threads,
                                    uint64_t* out);
B2Z_API b2z_status b2z_fr_lincomb3(uint64_t count, const uint64_t a[4], const uint64_t* x, const uint64_t b[4],
                                   const uint64_t* y, const uint64_t c[4], const uint64_t* z, uint32_t threads,
                                   uint64_t* out);
B2Z_API b2z_status b2z_fr_into_bigint(uint64_t count, const uint64_t* in, uint32_t threads, uint64_t* out);

/* ---- witness generation on the host, multithreaded (SURVEY.md 8(f) row f5; no GPU, no ctx) ---------------------
 * Once a proof takes tens of milliseconds the assignment itself is the next bottleneck.  The reference computes
 * witnesses during synthesis (ark-r1cs-std), next to two native helpers restated here: hasher() -- the Poseidon sponge
 * digest of a flattened matrix, absorb everything / squeeze one element
 * (src/arkworks/matrix_proof_of_work/hasher.rs:17-27) -- and mod_pow_generate_witnesses()
 * (src/arkworks/prime_snark/utils/modulo.rs:31-89).  The Poseidon parameters are ARGUMENTS (a Rust caller passes its
 * PoseidonConfig: full_rounds, partial_rounds, alpha, ark, mds, rate, capacity -- hashing_utils.rs:701-715); the
 * library carries no table.  All field elements: 4 x u64 Montgomery limbs, canonical (< r), else B2Z_EINVAL.       */
typedef struct b2z_poseidon_desc {
  uint32_t full_rounds;     /* even: half before and half after the partial rounds (8 in the reference)            */
  uint32_t partial_rounds;  /* S-box on state[0] only (29)                                                          */
  uint64_t alpha;           /* S-box exponent (17): left-to-right square-and-multiply, one witness per product      */
  uint32_t width;           /* rate + capacity, 2 .. 8 (3)                                                          */
  uint32_t rate;            /* (2)                                                                                  */
  uint32_t capacity;        /* (1): rate slots sit AFTER the capacity slots in the state                            */
  const uint64_t* ark;      /* (full_rounds + partial_rounds) x width round constants                               */
  const uint64_t* mds;      /* width x width, row-major                                                             */
} b2z_poseidon_desc;
/* PoseidonSponge::new(params).absorb(elems).squeeze_native_field_elements(1)[0] */
B2Z_API b2z_status b2z_poseidon_hash(const b2z_poseidon_desc* params, const uint64_t* elems, uint64_t count,
                                     uint64_t digest_out[4]);
/* Full assignment of the matrix-multiplication circuit for n x n inputs a, b (row-major)
 * (matrix_proof_of_work/constraints.rs:78-128: witnesses A, B; C = A B with one product witness per scalar product
 * and a zero-initialised sum witness per entry; public digests of A, B, C), in the variable order of this
 * repository's circuit builder (zksnark-finalproject_b200/circuits.py: matrix_circuit):
 *   [1, digest(A), digest(B), digest(C) | A | B | S-box witnesses of digest(A) | of digest(B) | n^2 zeros |
 *    per (i, j): sum witness (0), a_i0 b_0j .. a_i,n-1 b_n-1,j | S-box witnesses of digest(C)]
 * z_out: b2z_matrix_circuit_num_variables(params, n) elements, ready for b2z_groth16_prove_r1cs; B2Z_ESIZE when
 * z_capacity (in elements) is smaller.  threads: 0 = all hardware threads.  The digests of A and B are independent
 * sequential chains (one thread each) beside the n^3 products (the other threads); the digest of C follows.     */
B2Z_API uint64_t b2z_matrix_circuit_num_variables(const b2z_poseidon_desc* params, uint32_t n);
B2Z_API b2z_status b2z_matrix_circuit_witness(const b2z_poseidon_desc* params, uint32_t n, const uint64_t* a,
                                              const uint64_t* b, uint32_t threads, uint64_t* z_out,
                                              uint64_t z_capacity);
/* Assignment of the Fibonacci circuit (src/arkworks/constraints/fibbonaci.rs:22-48): [1, a, b, F(num_steps) | 0],
 * the result computed in Fr.                                                                                     */
B2Z_API b2z_status b2z_fibonacci_witness(const uint64_t a[4], const uint64_t b[4], uint64_t num_steps,
                                         uint64_t z_out[20]);
/* mod_pow_generate_witnesses(base, div, exp) for base, modulus < 2^63 and num_bits table rows (the reference
 * hard-codes 382): mod_pow_vals[i] = the i-th squaring of the chain power <- power^2 mod modulus, mod_vals[i] = the
 * running product after exponent bit i (least significant first; rows past the exponent's length repeat the result
 * with quotient 0), each row = (value lo, value hi, quotient lo, quotient hi, remainder) with value BEFORE the
 * reduction; bits[i] = exponent bit i; *result = base^exponent mod modulus.  exponent must fit num_bits.
 * (Where the reference's BigUint subtraction `cur_pow - 1` would panic -- cur_pow = 0 -- this returns the
 * arithmetic value.)                                                                                            */
B2Z_API b2z_status b2z_modpow_witnesses(uint64_t base, uint64_t modulus, uint64_t exponent, uint32_t num_bits,
                                        uint64_t* mod_vals /* num_bits x 5 */, uint64_t* mod_pow_vals /* num_bits x 5 */,
                                        uint8_t* bits /* num_bits */, uint64_t* result);

/* The prime route's native search (src/arkworks/backend/prime_snark.rs:60-70): for j = j_first .. j_last,
 * check_if_next_is_prime(x, j) (prime_snark/prime_circut.rs:165-195) until one succeeds --
 *   a_j = SHA-256(le32(x + j));  candidate = a_j mod 2^num_bits (utils/constants.rs: NUM_BITS = 20), quotient = a_j >> num_bits;
 *   a = Fr::from_le_bytes_mod_order(SHA-256(le32(x + j) || a_j || le64(j)));
 *   fermat_test(a, candidate) (fermat_circut.rs:131-141): bases SHA-256(le32(a) || le32(jj)) mod candidate for
 *   jj < k_bases (constants.rs: K = 3), "prime" when ANY base b satisfies b^(candidate-1) = 1 mod candidate.
 * The j are spread over `threads` host threads (0 = all); the SMALLEST successful j is returned, i.e. the reference's
 * loop exit.  *found = 0: none in the range, *out then describes j_last.  x: Fr, Montgomery limbs.  num_bits <= 62.
 * candidate = 0 (where the reference's BigUint division panics) counts as not prime.                              */
typedef struct b2z_prime_check {
  uint64_t j;
  uint8_t digest[32];      /* a_j, the bytes SHA-256 produced (IsPrimeStruct.0)                                   */
  int32_t is_prime;        /* IsPrimeStruct.1                                                                     */
  uint64_t quotient[4];    /* IsPrimeStruct.2.q, little-endian limbs                                              */
  uint64_t remainder;      /* IsPrimeStruct.2.remainder: the candidate                                            */
  uint64_t a[4];           /* IsPrimeStruct.3: canonical integer, little-endian limbs                             */
} b2z_prime_check;
B2Z_API b2z_status b2z_prime_search(const uint64_t x[4], uint64_t j_first, uint64_t j_last, uint32_t num_bits,
                                    uint32_t k_bases, uint32_t threads, b2z_prime_check* out, int32_t* found);
/* SHA-256 of a byte string (the `sha2` crate the native side of the prime route uses) */
B2Z_API void b2z_sha256(const uint8_t* data, uint64_t len, uint8_t digest_out[32]);

/* ---- measurement hooks ----------------------------------------------------------------
 * Phase timers use CUDA events recorded on the stream each kernel is launched on.
 * Phases (index into the arrays of b2z_profile_read, length B2Z_PHASE_COUNT):
 *   0 NTT pass kernels (units: field elements)   1 witness-map pointwise (elements)
 *   2 MSM digits + counting sort (scalars)       3 MSM bucket accumulation G1 (mixed adds)
 *   4 MSM bucket accumulation G2 (mixed adds)    5 MSM partial lists / bucket reduction / combine
 *   6 constraint-row evaluation (CSR SpMV of A, B, C against z)
 *   7 the accumulation launches of 3 / 4 that took the batched-affine kernel (counted there too)   */
#define B2Z_PHASE_COUNT 8
B2Z_API b2z_status b2z_profile_enable(b2z_ctx* ctx, int on);
B2Z_API b2z_status b2z_profile_read(b2z_ctx* ctx, double* ms, uint64_t* launches, uint64_t* units, int reset);
/* timeline of the recorded spans relative to the first one (development aid); returns the count */
B2Z_API int b2z_profile_spans(b2z_ctx* ctx, int max_spans, int* phase, double* start_ms, double* stop_ms);
/* kernels launched through this context since its creation */
B2Z_API uint64_t b2z_kernel_launches(const b2z_ctx* ctx);
/* measured 32-bit multiply-add issue rates of the device (ops/s): plain IMAD and the
 * carry-chained 32x32+64 wide form the field arithmetic is built from               */
B2Z_API b2z_status b2z_measure_int_peak(b2z_ctx* ctx, double* imad_per_s, double* imad_wide_per_s);

/* ---- Point-sharded proof with a DISTRIBUTED witness map (SURVEY.md 8(e)) -------------------------------------
 * With b2z_groth16_prove_partial every shard repeats the whole witness map (8.4 of the 25 ms a shard-of-8 takes
 * at 2^22).  Here the three input transforms are done once per box:
 *   - every rank:        b2z_groth16_shard_begin(ctx, pk_shard, r1cs, z, r, s)
 *        starts everything that depends on z only (four sorts, the B2 / A / B1 / L accumulations) and returns
 *        while the GPU is busy;
 *   - rank j in {0,1,2}: b2z_r1cs_coset_evals(ctx, r1cs, j, z, d_out)
 *        rows of matrix j (0 = A, 1 = B, 2 = C) against z, then inverse transform + coset transform, into a
 *        caller-owned DEVICE buffer of 2^log_n x 32 bytes; returns when d_out is complete.  The caller sends it to
 *        the other ranks (NCCL broadcast, peer copy ...): the library links no communication runtime.  An owner
 *        should call this BEFORE shard_begin -- the accumulations fill the GPU and would starve the transform
 *        every other rank is waiting for;
 *   - every rank:        b2z_groth16_shard_finish(ctx, pk_shard, d_a, d_b, d_c, partial_out)
 *        pointwise quotient, last transform, this shard's H sum, host epilogue: B2Z_PARTIAL_BYTES as from
 *        b2z_groth16_prove_partial (d_a is clobbered).  Combine with b2z_groth16_combine.
 * z: the assignment for the FIRST of these calls of a proof (it is uploaded once), NULL afterwards -- NULL is only
 * accepted inside one proof: shard_finish invalidates the uploaded assignment, so a mis-sequenced call fails with
 * B2Z_EINVAL instead of proving a stale one.  A rank must not start another proof on the same key / r1cs (nor free
 * the r1cs) before shard_finish.                                                                                  */
B2Z_API b2z_status b2z_groth16_shard_begin(b2z_ctx* ctx, const b2z_pk* pk, b2z_r1cs* r1cs, const uint64_t* z,
                                           const uint64_t r[4], const uint64_t s[4]);
B2Z_API b2z_status b2z_r1cs_coset_evals(b2z_ctx* ctx, b2z_r1cs* r1cs, uint32_t which, const uint64_t* z,
                                        uint64_t* d_out);
B2Z_API b2z_status b2z_groth16_shard_finish(b2z_ctx* ctx, const b2z_pk* pk, uint64_t* d_a, const uint64_t* d_b,
                                            const uint64_t* d_c, uint8_t* partial_out);

/* ---- ONE proof by 2, 4 or 8 GPUs of a box with the WITNESS MAP ITSELF tile-sharded (SURVEY.md 8(e)) -----------
 * One rank per GPU (a process per GPU under torchrun, or a host thread per GPU in one process).  Every rank holds
 * shard `rank` of the key (b2z_pk_upload_shard) and the matrices.  Per proof:
 *   - each rank moves 1 / W of the assignment over PCIe and copies that slice into the peers' memory over NVLink;
 *   - the witness map runs on n / W elements per rank: the transform's stages are split between a column-owned
 *     and a row-owned layout, and each layout change (an all-to-all transpose) is fused into the STORE of the
 *     pass before it -- the kernel writes its output tile straight into the peers' buffers over NVLink
 *     (3 exchanges per proof, 3 x n x 32 / W bytes per rank at most);
 *   - rank k ends with coefficients [n k / W, n (k + 1) / W) of h (bit-reversed order) = exactly the h bases of
 *     its key shard, so the five MSM accumulations follow back to back with no further data exchange;
 *   - the 1344-byte partial sums meet in a caller-provided SHARED HOST buffer and every rank returns the proof.
 * The library links no communication runtime: peers are attached either by CUDA IPC handle (another process)
 * or by plain device pointer (same process), and ranks synchronise by a host barrier on the shared buffer
 * (b2z_dist_shared_bytes(world) bytes, zero-initialised, visible to all ranks: POSIX shared memory between
 * processes, ordinary memory between threads).  All ranks must call b2z_dist_prove for the same proof with the
 * same r, s; the call returns on every rank with the same 192 bytes.
 *   z: the full assignment (host or device pointer; each rank reads only its slice), or, with
 *      z_is_full_device_copy != 0, a device-resident full copy per rank (no exchange).
 * B2Z_ESIZE from b2z_dist_create: the domain is too small to tile (fall back to b2z_groth16_prove_partial_r1cs). */
typedef struct b2z_dist b2z_dist;
B2Z_API uint64_t b2z_dist_shared_bytes(uint32_t world);
B2Z_API b2z_status b2z_dist_create(b2z_ctx* ctx, const b2z_pk* pk_shard, b2z_r1cs* r1cs, uint32_t rank, uint32_t world,
                                   void* shared_host, b2z_dist** out);
B2Z_API void b2z_dist_destroy(b2z_ctx* ctx, b2z_dist* dist);
/* this rank's exchange region: ipc_handle (64 bytes, cudaIpcMemHandle_t) and / or its device pointer */
B2Z_API b2z_status b2z_dist_export(b2z_ctx* ctx, b2z_dist* dist, uint8_t ipc_handle[64], void** device_ptr);
/* make rank `peer`'s region reachable: exactly one of ipc_handle (other process) / device_ptr (same process) */
B2Z_API b2z_status b2z_dist_attach(b2z_ctx* ctx, b2z_dist* dist, uint32_t peer, const uint8_t* ipc_handle,
                                   void* device_ptr);
/* host only (no GPU, no ctx): the last step of b2z_dist_prove on its own -- this rank's B2Z_PARTIAL_BYTES go into
 * the shared buffer, a barrier, every rank combines all `world` partials into the proof, a second barrier.
 * *epoch: this rank's barrier counter (start at 0; same call sequence on every rank).                          */
B2Z_API b2z_status b2z_dist_combine_shared(void* shared_host, uint32_t rank, uint32_t world, uint32_t* epoch,
                                           const uint8_t* my_partial, uint8_t proof_out[192]);
B2Z_API b2z_status b2z_dist_prove(b2z_ctx* ctx, b2z_dist* dist, const uint64_t* z, int z_is_full_device_copy,
                                  const uint64_t r[4], const uint64_t s[4], uint8_t proof_out[192]);

/* Page-lock caller-owned host memory (cudaHostRegister) so that the per-proof upload of the assignment runs at
 * PCIe speed instead of through the driver's staging buffer (61 MB of z at 2^22: ~1.2 ms instead of ~4 ms).  The
 * caller keeps ownership; unregister before freeing.  A Rust caller registers the Vec<Fr> it reuses per request. */
B2Z_API b2z_status b2z_host_register(b2z_ctx* ctx, void* ptr, uint64_t bytes);
B2Z_API b2z_status b2z_host_unregister(b2z_ctx* ctx, void* ptr);

/* ---- host-side self checks (no GPU needed) -------------------------------------------
 * The limb algorithms of the device code are written against a carry-flag
 * abstraction that also runs on the host; these entry points let the CPU-only test
 * suite check them against the oracle.  op: 0 mul, 1 add, 2 sub, 3 canonical form,
 * 4 inverse.  field: 0 = Fr (8 x u32), 1 = Fq (12 x u32); operands lazy (< 2p).      */
B2Z_API int b2z_host_field_op(int field, int op, const uint32_t* a, const uint32_t* b, uint32_t* out);
/* Fq inversion by division steps (csrc/inv_gcd.cuh, the shared inversion of the batched-affine bucket accumulation):
 * a, out = 12 x u32 Montgomery limbs (a lazy, out canonical; 0 -> 0); returns the number of 30-step batches used. */
B2Z_API int b2z_host_fq_inv_gcd(const uint32_t* a, uint32_t* out);
/* The batched-affine bucket accumulation (csrc/accum_affine.cuh) run on the host, one emulated thread per segment:
 * points = affine bases (24 / 48 u32 each), sorted = point references ordered by bucket (bit 31 = negated),
 * offsets[nbuckets + 1] = start of every bucket in `sorted`, cap = reserved (pass 0).
 * Returns the number of buckets whose sum (bucket + partial entries) differs from the XYZZ running sum.
 * maxrun_out[7]: the run bound, then completed rounds, batched additions, doublings among them, division-free
 * pairs + carried entries, abandoned rounds, mixed additions of the XYZZ finish.                                */
B2Z_API int b2z_host_accum_affine(int group /*1|2*/, const uint32_t* points, const uint32_t* sorted,
                                  const uint32_t* offsets, uint32_t nbuckets, uint32_t nseg, uint32_t cap,
                                  uint32_t* maxrun_out);
/* sum of n affine points (Montgomery limbs, 24 / 48 u32 each; neg[i] != 0 negates) with the
 * device's XYZZ mixed-addition code; out = affine sum, returns 1 if the sum is the identity. */
B2Z_API int b2z_host_point_sum(int group /*1|2*/, const uint32_t* points, const uint8_t* neg, uint32_t n,
                               uint32_t* out_affine);
/* signed digits of a canonical scalar as the MSM kernels see them; returns the window count */
B2Z_API uint32_t b2z_host_msm_digits(const uint32_t scalar[8], uint32_t c, int32_t* digits /* >= 64 */);
B2Z_API uint32_t b2z_host_msm_window_bits(uint64_t n, int precomputed);
/* the host-side last step of an MSM (csrc/host_fq.hpp, what the prover's epilogue runs): planes[0] +
 * 2^chunk_log * sum_{k>=1} 2^(k-1) planes[k] for nplanes XYZZ points in the device layout (48 / 96 u32 each),
 * serialised compressed (48 / 96 bytes) into out                                                                */
B2Z_API int b2z_host_planes_horner(int group /*1|2*/, const uint32_t* planes_xyzz, uint32_t nplanes, uint32_t chunk_log,
                                   uint8_t* out);
/* b2z_groth16_verify_batch's per-proof device code (csrc/pairing.cuh: decode, Miller loop, final exponentiation) run
 * on the host for one proof, with the batch call's call-level checks and statuses; *result = 1 / 0 / -1.          */
B2Z_API b2z_status b2z_host_verify_one(const uint8_t* pvk, uint64_t pvk_len, const uint64_t* public_inputs,
                                       uint64_t num_inputs, const uint8_t proof[192], int32_t* result);
/* pairing.cuh's tower pieces next to csrc/host_pairing.hpp's on canonical Montgomery limbs (Fq12 = 144 u32 in tower
 * order c0.c0.c0 .. c1.c2.c1, Fq2 = 24 u32): op 0 a * b, 1 a^2, 2 a^q, 3 final exponentiation, 4 an Fq2 square root
 * (the root that is not lexicographically largest).  out_dev / out_host: the two results, canonical.  Returns 0; for
 * op 3, 1 when a != 0 (-2 when the sides disagree); for op 4, (root on the device side) + 2 (root on the host side). */
B2Z_API int b2z_host_pairing_op(int op, const uint32_t* a, const uint32_t* b, uint32_t* out_dev, uint32_t* out_host);

#ifdef __cplusplus
}
#endif
#endif /* B200ZK_H_ */
