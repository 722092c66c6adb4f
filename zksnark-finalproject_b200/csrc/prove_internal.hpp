// The proving key and the phases of a proof on it, shared by prove.cu, r1cs.cu and setup.cu.
#pragma once
#include "common.hpp"
#include "ec.cuh"
#include "msm.hpp"

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

// ---------------------------------------------------------------------------
// Proving key
// ---------------------------------------------------------------------------
constexpr uint32_t kCycBlock = 64;   // variables per block of the block-cyclic point sharding

// local variable j of a block-cyclic shard -> global variable index
__host__ __device__ inline uint64_t cyc_global(uint64_t j, uint32_t rank, uint32_t world) {
  return ((j / kCycBlock) * world + rank) * kCycBlock + (j % kCycBlock);
}

// Which part of a key a handle holds: a whole key, or one shard of it.
// shard: `ma` variables of the a/b queries -- either the contiguous range [lo, lo+ma) (cyc_world == 0) or,
// block-cyclic, the blocks cyc_rank, cyc_rank + cyc_world, ... of kCycBlock variables (balanced whatever the
// witness structure: Groth16 assignments have long stretches of small / Boolean values); the first l_skip of
// them are instance variables (not in l_query), ml = ma - l_skip; bit-reversed h positions [h_lo, h_lo+hn);
// alpha/beta/delta terms on shard 0 only
struct PkShard {
  uint32_t log_n = 0;
  uint64_t m = 0, l = 0;
  uint32_t lo = 0, ma = 0, l_skip = 0, ml = 0, h_lo = 0, hn = 0, with_vk = 1;
  uint32_t cyc_world = 0, cyc_rank = 0;
  // global index of the shard's local variable j
  __host__ __device__ uint64_t var(uint64_t j) const { return cyc_world ? cyc_global(j, cyc_rank, cyc_world) : lo + j; }
  // every variable, every h position and the alpha/beta/delta terms: not a shard
  bool whole() const { return with_vk && cyc_world == 0 && lo == 0 && ma == m && hn == (1ull << log_n); }
};

// The sharding rule of every key handle (b2z_pk_upload / _slice / _shard, b2z_groth16_setup[_shard]): the slice
// [from, to) of den.  Variables: the contiguous range [m from/den, m to/den), or, for cyc_world > 1, the block-cyclic
// variables of rank cyc_rank -- contiguous after all when l > kCycBlock (the instance variables must sit in block 0).
// h positions: [n from/den, n to/den) of the bit-reversed order.  The slice with from == 0 keeps alpha/beta/delta.
inline PkShard pk_shard(uint32_t log_n, uint64_t m, uint64_t l, uint32_t from, uint32_t to, uint32_t den,
                        uint32_t cyc_rank, uint32_t cyc_world) {
  PkShard S;
  S.log_n = log_n;
  S.m = m;
  S.l = l;
  if (cyc_world > 1 && l <= kCycBlock) {
    uint64_t ma = 0;
    for (uint64_t b = cyc_rank; b * kCycBlock < m; b += cyc_world)
      ma += m - b * kCycBlock < kCycBlock ? m - b * kCycBlock : kCycBlock;
    S.cyc_world = cyc_world; S.cyc_rank = cyc_rank;
    S.lo = 0; S.ma = (uint32_t)ma;
    S.l_skip = cyc_rank == 0 ? (uint32_t)(l < ma ? l : ma) : 0;
  } else {
    const uint64_t lo = m * from / den, hi = m * to / den;
    const uint64_t l_lo = lo > l ? lo : l;             // first witness variable in the slice
    S.lo = (uint32_t)lo; S.ma = (uint32_t)(hi - lo);
    S.l_skip = (uint32_t)((l_lo < hi ? l_lo : hi) - lo);
  }
  S.ml = S.ma - S.l_skip;
  const uint64_t n = 1ull << log_n, h_lo = n * from / den, h_hi = n * to / den;
  S.h_lo = (uint32_t)h_lo; S.hn = (uint32_t)(h_hi - h_lo);
  S.with_vk = from == 0 ? 1u : 0u;
  return S;
}

// A key's five base sets in device memory (points + identity bitmap words), the layout b2z_pk_upload assembles, for
// the shard's variables and h positions; the alpha/beta/delta terms only when S.with_vk:
// a, b1, b2: ma (+ 2) points [query | alpha_1 delta_1] / [query | beta_1 delta_1] / [query | beta_2 delta_2];
// l: ml (+ 1) points [l_query | delta_1]; h: hn points of h_query in bit-reversed order, position n - 1 the flagged
// identity.
struct PkDeviceSets {
  const G1::Affine *a, *b1, *l, *h;
  const G2::Affine* b2;
  const uint32_t *a_words, *b1_words, *l_words, *h_words, *b2_words;
};
// b2z_pk_upload's rule for precomputed window copies: `num` / `den` of a whole key's copies fit in half the free
// device memory (a shard of `world`: 1 / world)
bool pk_precompute_fits_slice(uint32_t log_n, uint64_t m, uint64_t l, uint32_t num, uint32_t den);
// the key handle of shard S for its sets (copied; the caller keeps its buffers); `pre` from pk_precompute_fits_slice
b2z_pk* pk_from_device_sets(Ctx& c, const PkShard& S, const PkDeviceSets& sets, bool pre);

// The five MSMs of a proof, the G1 ones first.  (The partial sums leave in the order A | sA | rB1 | L | H | B,
// B2Z_PARTIAL_BYTES.)
enum Sum { SUM_A, SUM_B1, SUM_L, SUM_H, SUM_B, SUM_COUNT };

// Where one MSM of a proof runs and what it leaves.
struct ProofSum {
  int slot = 0;                      // MSM scratch arena
  cudaStream_t stream = nullptr;     // its accumulation (and, but for H, its sort); H: set by proof_h_sort
  uint32_t tail = 0;                 // its extra scalars: PkImpl::tail + this (not H)
  void* d_result = nullptr;          // one XYZZ point (G2 for B)
  MsmHostPlanes planes;              // its bit-plane sums, for the Horner pass on the host
  cudaEvent_t accum = nullptr;       // accumulation kernel done (the next sum of the chain waits for it; not H)
  cudaEvent_t done = nullptr;        // planes copied to the host (not H: proof_end synchronises its stream)
  cudaEvent_t sorted = nullptr;      // L only: sort done (the G2 accumulation waits for it)
  template <class C> typename C::Xyzz* result() const { return static_cast<typename C::Xyzz*>(d_result); }
};

struct PkImpl : PkShard {
  // A key handle holds per-proof scratch (below), so it belongs to exactly ONE context: the one it was
  // uploaded through.  Every entry point checks this and returns B2Z_EINVAL for a foreign context.
  const Ctx* owner = nullptr;
  bool* assignment_flag = nullptr;   // b2z_groth16_shard_begin .. shard_finish window (r1cs.cu)
  MsmBases<G1> a_set;          // [a_query  | alpha_1 delta_1]
  MsmBases<G1> b1_set;         // [b_g1     | beta_1  delta_1]
  MsmBases<G1> l_set;          // [l_query  | delta_1]
  MsmBases<G1> h;              // h_query, bit-reversed order, padded to n (this shard's positions)
  MsmBases<G2> g2;             // [b_g2     | beta_2  delta_2]
  // per-proof device scratch
  DevBuf<FrEl> ea, eb, ec, z, zc, hc, tail;
  DevBuf<G1::Xyzz> g1_out;     // results of the G1 sums, indexed by Sum (s*A and r*B1 are made on the host)
  DevBuf<G2::Xyzz> g2_out;     // result of B
  uint32_t* h_out = nullptr;   // pinned: B2Z_PARTIAL_BYTES
  uint32_t* h_planes = nullptr;   // pinned: bit-plane sums of the five MSMs (host-side Horner, msm.hpp)
  ProofSum sums[SUM_COUNT];
  FrEl r_c, s_c;                  // the proof's r, s as canonical integers (proof_begin -> proof_end)
  cudaEvent_t ev_z = nullptr;
  cudaEvent_t ev_wm = nullptr;       // witness-map transforms of the proof in flight are done (gates the first accumulation)
  ~PkImpl() {
    if (h_out) cudaFreeHost(h_out);
    if (h_planes) cudaFreeHost(h_planes);
    if (ev_z) cudaEventDestroy(ev_z);
    for (ProofSum& S : sums)
      for (cudaEvent_t e : {S.accum, S.done, S.sorted})
        if (e) cudaEventDestroy(e);
    if (ev_wm) cudaEventDestroy(ev_wm);
  }
};

// the key behind a handle; B2Z_EINVAL naming `who` when it is NULL or was uploaded through another context
PkImpl& pk_of(Ctx& c, const b2z_pk* pk, const char* who);

// ---------------------------------------------------------------------------
// A proof on a key (a whole key or one shard of it) in five phases that share the key's scratch.  Each driver calls
// them around its own witness map: proof_begin first, proof_end last, proof_h_finish after proof_h_sort (its stream)
// and proof_accums (the event it chains after).
//   proof_begin     everything that depends on z only: the tail scalars {1, r, 1, s, -rs}, this shard's variables
//                   of z (Montgomery form, d_z) as canonical integers, and the sorts of A, B (G2), B1 and L
//   proof_h_sort    this shard's h coefficients (bit-reversed positions [h_lo, h_lo + hn), Montgomery form, d_h) to
//                   canonical form, then the sort of H, on `st`; H accumulates on `st` too
//   proof_accums    the accumulations A -> B1 -> B -> L, chained; the first waits for `gate` (nullptr: none)
//   proof_h_finish  the accumulation of H, after L's
//   proof_end       waits for the five sums and does the host epilogue: XYZZ partial sums A, s*A, r*B1, L, H (G1)
//                   and B (G2) in partial_out (B2Z_PARTIAL_BYTES, host memory)
void proof_begin(Ctx& c, PkImpl& P, const FrEl* d_z, const uint64_t r[4], const uint64_t s[4]);
void proof_h_sort(Ctx& c, PkImpl& P, const FrEl* d_h, cudaStream_t st);
void proof_accums(Ctx& c, PkImpl& P, cudaEvent_t gate);
void proof_h_finish(Ctx& c, PkImpl& P);
void proof_end(Ctx& c, PkImpl& P, uint8_t* partial_out);

// the single-GPU proof from device-resident a/b/c evaluations (d_a is clobbered) and assignment: this shard's partial
// sums; prove_device: the 192 proof bytes, on a whole key only (B2Z_EINVAL otherwise)
void prove_partial_device(Ctx& c, PkImpl& P, FrEl* d_a, FrEl* d_b, FrEl* d_c, const FrEl* d_z, const uint64_t r[4],
                          const uint64_t s[4], uint8_t* partial_out);
void prove_device(Ctx& c, PkImpl& P, FrEl* d_a, FrEl* d_b, FrEl* d_c, const FrEl* d_z, const uint64_t r[4],
                  const uint64_t s[4], uint8_t proof_out[192]);
// host epilogue of a proof: sum the partials of `world` shards, normalise, serialise
void combine_partials(const uint8_t* partials, uint32_t world, uint8_t proof_out[192]);
}  // namespace b2z
