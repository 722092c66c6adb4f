// Entry points of prove.cu and r1cs.cu used by the other translation units (r1cs.cu, setup.cu).
#pragma once
#include "common.hpp"
#include "ec.cuh"

struct b2z_pk;
struct b2z_r1cs;

namespace b2z {
// one constraint matrix on the device, CSR as uploaded (column indices < num_variables, Montgomery coefficients)
struct CsrDev {
  DevBuf<uint32_t> row_ptr, cols;
  DevBuf<FrEl> coeffs;
};
// the matrices of an uploaded r1cs; B2Z_EINVAL when the handle belongs to another context
struct R1csView {
  uint64_t nc, l, m;
  uint32_t log_n;
  const CsrDev* mat;   // A, B, C
};
R1csView r1cs_view(Ctx& c, b2z_r1cs* r, const char* who);

// A whole key's five base sets in device memory (points + identity bitmap words), the layout b2z_pk_upload assembles:
// a, b1, b2: m + 2 points [query | alpha_1 delta_1] / [query | beta_1 delta_1] / [query | beta_2 delta_2];
// l: m - l + 1 points [l_query | delta_1]; h: n points, h_query in bit-reversed order, position n - 1 the flagged identity.
struct PkDeviceSets {
  const G1::Affine *a, *b1, *l, *h;
  const G2::Affine* b2;
  const uint32_t *a_words, *b1_words, *l_words, *h_words, *b2_words;
};
// b2z_pk_upload's rule for precomputed window copies: they fit in half the free device memory
bool pk_precompute_fits(uint32_t log_n, uint64_t m, uint64_t l);
// the key handle for those sets (copied; the caller keeps its buffers); `pre` from pk_precompute_fits
b2z_pk* pk_from_device_sets(Ctx& c, uint32_t log_n, uint64_t m, uint64_t l, const PkDeviceSets& sets, bool pre);
bool pk_matches(const b2z_pk* pk, uint32_t log_n, uint64_t m, uint64_t l);
// whole-key proof from device-resident a/b/c evaluations (clobbered) and assignment
void prove_on_device_buffers(Ctx& c, const b2z_pk* pk, FrEl* d_a, FrEl* d_b, FrEl* d_c, const FrEl* d_z,
                             const uint64_t r[4], const uint64_t s[4], uint8_t proof_out[192]);
// the same for one shard of a key: B2Z_PARTIAL_BYTES of partial sums
void prove_partial_on_device_buffers(Ctx& c, const b2z_pk* pk, FrEl* d_a, FrEl* d_b, FrEl* d_c, const FrEl* d_z,
                                     const uint64_t r[4], const uint64_t s[4], uint8_t* partial_out);
// the same in two calls (sharded prover with a distributed witness map): z-only work first (returns while the
// GPU is busy), then quotient + H + host epilogue from the three COSET evaluation vectors (d_a is clobbered)
void prove_begin_on(Ctx& c, const b2z_pk* pk, const FrEl* d_z, const uint64_t r[4], const uint64_t s[4]);
// tile-sharded prover (r1cs.cu: b2z_dist_*): z-only sorts; the H sort from this shard's chunk of h; the chained
// accumulations + host epilogue once `ready` has fired
void prove_begin_sorts_on(Ctx& c, const b2z_pk* pk, const FrEl* d_z, const uint64_t r[4], const uint64_t s[4]);
uint32_t pk_h_chunk(const b2z_pk* pk, uint32_t* h_lo);
void prove_dist_h_sort_on(Ctx& c, const b2z_pk* pk, const FrEl* d_h, cudaStream_t st);
void prove_dist_finish_on(Ctx& c, const b2z_pk* pk, cudaEvent_t wm_done, cudaStream_t h_st, uint8_t* partial_out);
void combine_partials_host(const uint8_t* partials, uint32_t world, uint8_t proof_out[192]);
// remembers where the "assignment uploaded" flag of the r1cs used by shard_begin lives; prove_finish_on clears it
void pk_bind_assignment_flag(const b2z_pk* pk, bool* flag);
void prove_finish_on(Ctx& c, const b2z_pk* pk, FrEl* d_a, const FrEl* d_b, const FrEl* d_c, uint8_t* partial_out);
}  // namespace b2z
