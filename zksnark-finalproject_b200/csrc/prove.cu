// Groth16 prover assembly -- replaces ark-groth16 0.4's create_proof_with_reduction /
// create_proof_with_assignment minus circuit synthesis (reference call sites:
// src/arkworks/backend/fibbonaci_handler.rs:110, matrix_proof.rs:139-140,
// prime_snark.rs:119; equations: SURVEY.md A.4):
//
//   A  = alpha_1 + sum z_i a_i + r delta_1
//   B  = beta_2  + sum z_i b2_i + s delta_2          B1 = beta_1 + sum z_i b1_i + s delta_1
//   C  = s A + r B1 - r s delta_1 + sum_{i>=l} z_i l_i + sum h_i hq_i
//
// Five MSMs on five streams, every "+ constant" folded into them as extra (point, scalar) pairs:
//   A   : G1 [a_query  | alpha_1 delta_1]   x [z | 1 r]
//   B1  : G1 [b_g1     | beta_1  delta_1]   x [z | 1 s]
//   L   : G1 [l_query  | delta_1]           x [z_{>=l} | -rs]
//   H   : G1 h_query in bit-reversed order  x h   (the order the DIF witness map leaves h in)
//   B   : G2 [b_g2     | beta_2  delta_2]   x [z | 1 s]
// All of them read z as it is (small / Boolean witness values keep their few non-zero digits).
// s*A and r*B1 -- 255-bit double-and-add on freshly computed points, the one inherently serial
// piece of arkworks' formulation -- are done where arkworks does them, on the host, as soon as A
// and B1 have been copied back and WHILE the GPU is still accumulating L and H (0.2 ms each on a
// CPU core).  Schedule: light work first (scalar prep, all sorts, witness map), then the
// GPU-filling accumulations chained back to back, each tail overlapping the next accumulation.
// The host finishes with a few point additions, three affine normalisations and the
// serialization (host_fq.hpp).  r = 0: r*B1 is the identity, exactly arkworks' special case.
#include <cstring>

#include "api_glue.hpp"
#include "host_fq.hpp"
#include "msm.hpp"
#include "prove_internal.hpp"

namespace b2z {

namespace {

// dst[p] = src[bitrev(p)] when that index exists, else identity (flagged)
__global__ void permute_bitrev_g1_kernel(const G1::Affine* __restrict__ src, const uint32_t* __restrict__ src_inf,
                                         uint32_t n_src, uint32_t log_n, G1::Affine* dst, uint32_t* dst_flags) {
  const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= (1u << log_n)) return;
  const uint32_t j = log_n == 0 ? 0 : (__brev(p) >> (32 - log_n));
  bool inf = j >= n_src;
  if (!inf && src_inf != nullptr) inf = (src_inf[j >> 5] >> (j & 31)) & 1;
  if (inf) {
    G1::Affine z;
    z.x = Fq::zero();
    z.y = Fq::zero();
    dst[p] = z;
  } else {
    dst[p] = src[j];
  }
  dst_flags[p] = inf ? 1u : 0u;
}

constexpr uint32_t kCycBlock = 64;   // variables per block of the block-cyclic point sharding

// local variable j of a block-cyclic shard -> global variable index
__host__ __device__ inline uint64_t cyc_global(uint64_t j, uint32_t rank, uint32_t world) {
  return ((j / kCycBlock) * world + rank) * kCycBlock + (j % kCycBlock);
}
// zc[j] = canonical integer of z[global(j)]: this shard's MSM scalars
__global__ void fr_from_mont_cyclic_kernel(const FrEl* __restrict__ z, FrEl* zc, uint32_t count, uint32_t rank,
                                           uint32_t world) {
  const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= count) return;
  zc[j] = Fr::from_mont(z[cyc_global(j, rank, world)]);
}

FrEl fr_load_host(const uint64_t v[4]) {
  FrEl x;
  std::memcpy(x.l, v, 32);
  return x;
}

}  // namespace

// ---------------------------------------------------------------------------
// Proving key
// ---------------------------------------------------------------------------
// The five MSMs of a proof, the G1 ones first.  (The partial sums leave in the order A | sA | rB1 | L | H | B,
// B2Z_PARTIAL_BYTES.)
enum Sum { SUM_A, SUM_B1, SUM_L, SUM_H, SUM_B, SUM_COUNT };

// Where one MSM of a proof runs and what it leaves.
struct ProofSum {
  int slot = 0;                      // MSM scratch arena
  cudaStream_t stream = nullptr;     // its accumulation (and, but for H, its sort)
  uint32_t tail = 0;                 // its extra scalars: PkImpl::tail + this (not H)
  void* d_result = nullptr;          // one XYZZ point (G2 for B)
  MsmHostPlanes planes;              // its bit-plane sums, for the Horner pass on the host
  cudaEvent_t accum = nullptr;       // accumulation kernel done (the next sum of the chain waits for it; not H)
  cudaEvent_t done = nullptr;        // planes copied to the host (not H: prove_end synchronises its stream)
  cudaEvent_t sorted = nullptr;      // L only: sort done (the G2 accumulation waits for it)
  template <class C> typename C::Xyzz* result() const { return static_cast<typename C::Xyzz*>(d_result); }
};

struct PkImpl {
  // A key handle holds per-proof scratch (below), so it belongs to exactly ONE context: the one it was
  // uploaded through.  Every entry point checks this and returns B2Z_EINVAL for a foreign context.
  const Ctx* owner = nullptr;
  bool* assignment_flag = nullptr;   // b2z_groth16_shard_begin .. shard_finish window (r1cs.cu)
  uint32_t log_n = 0;
  uint64_t m = 0, l = 0;
  // shard: `ma` variables of the a/b queries -- either the contiguous range [lo, lo+ma) (cyc_world == 0) or,
  // block-cyclic, the blocks cyc_rank, cyc_rank + cyc_world, ... of kCycBlock variables (balanced whatever the
  // witness structure: Groth16 assignments have long stretches of small / Boolean values); the first l_skip of
  // them are instance variables (not in l_query), ml = ma - l_skip; bit-reversed h positions [h_lo, h_lo+hn);
  // alpha/beta/delta terms on shard 0 only
  uint32_t lo = 0, ma = 0, l_skip = 0, ml = 0, h_lo = 0, hn = 0, with_vk = 1;
  uint32_t cyc_world = 0, cyc_rank = 0;
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
  FrEl r_c, s_c;                  // the proof's r, s as canonical integers (prove_begin -> prove_end)
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

namespace {

// copies `count` points (+ identity bits) from host arrays into dst[at ...)
template <class Affine>
void stage_points(Affine* d_dst, std::vector<uint32_t>& words, uint64_t at, const uint64_t* pts, const uint8_t* inf,
                  uint64_t count, cudaStream_t st) {
  if (count == 0) return;
  B2Z_CUDA(cudaMemcpyAsync(d_dst + at, pts, count * sizeof(Affine), cudaMemcpyHostToDevice, st));
  if (inf != nullptr)
    for (uint64_t i = 0; i < count; i++)
      if ((inf[i >> 3] >> (i & 7)) & 1) words[(at + i) >> 5] |= 1u << ((at + i) & 31);
}

size_t pk_precompute_bytes(const b2z_pk_desc* d) {
  auto cost = [](uint64_t n, size_t pt) {
    if (n == 0) return (size_t)0;
    const uint32_t c = msm_pick_c(n, true);
    return (size_t)n * pt * msm_windows(c);
  };
  const uint64_t n = 1ull << d->log_domain;
  return 2 * cost(d->num_variables + 2, 96) + cost(d->num_variables - d->num_instance + 1, 96) +
         cost(d->num_variables + 2, 192) + cost(n, 96);
}

template <class C>
void msm_entry(Ctx& c, const uint64_t* bases, const uint8_t* inf_bitmap, const uint64_t* scalars, uint64_t n,
               uint64_t* out_xyz) {
  using Affine = typename C::Affine;
  using Xyzz = typename C::Xyzz;
  constexpr int kLimbs = sizeof(Affine) / 16;   // u64 limbs per coordinate (6 or 12)
  B2Z_REQUIRE(out_xyz != nullptr, B2Z_EINVAL, "msm: out is NULL");
  B2Z_REQUIRE(n == 0 || (bases != nullptr && scalars != nullptr), B2Z_EINVAL, "msm: NULL input");
  B2Z_REQUIRE(n < (1ull << 28), B2Z_ESIZE, "msm: more than 2^28 points in one call");
  // The signed-window recoding covers 255 bits (Fr::MODULUS_BIT_SIZE, what msm_bigint itself assumes): a scalar with
  // bit 255 set would index past the bucket array.  into_bigint() of an Fr element never has it; reject anything else.
  for (uint64_t i = 0; i < n; i++)
    B2Z_REQUIRE((scalars[4 * i + 3] >> 63) == 0, B2Z_EINVAL,
                "msm: scalar >= 2^255 (scalars must be canonical Fr bigints, i.e. into_bigint())");
  cudaStream_t st = c.stream;
  // identity as arkworks represents it: (1, 1, 0), Montgomery limbs
  std::memset(out_xyz, 0, 3 * kLimbs * 8);
  std::memcpy(out_xyz, host::kOne, 48);
  std::memcpy(out_xyz + kLimbs, host::kOne, 48);
  if (n == 0) return;
  MsmBases<C> B;
  {
    DevBuf<Affine> d(n);
    std::vector<uint32_t> words((n + 31) / 32, 0u);
    stage_points<Affine>(d.p, words, 0, bases, inf_bitmap, n, st);
    DevBuf<uint32_t> dinf;
    if (inf_bitmap != nullptr) {
      dinf.alloc(words.size());
      B2Z_CUDA(cudaMemcpyAsync(dinf.p, words.data(), words.size() * 4, cudaMemcpyHostToDevice, st));
    }
    msm_bases_build<C>(&c, B, d.p, dinf.p, (uint32_t)n, /*precompute=*/false, 0, st);
    B2Z_CUDA(cudaStreamSynchronize(st));
  }
  DevBuf<FrEl> ds(n);
  B2Z_CUDA(cudaMemcpyAsync(ds.p, scalars, n * sizeof(FrEl), cudaMemcpyHostToDevice, st));
  DevBuf<Xyzz> res(1);
  msm_run<C>(&c, 0, B, ds.p, (uint32_t)n, nullptr, res.p, st);
  uint32_t h_res[sizeof(Xyzz) / 4];
  B2Z_CUDA(cudaMemcpyAsync(h_res, res.p, sizeof(Xyzz), cudaMemcpyDeviceToHost, st));
  B2Z_CUDA(cudaStreamSynchronize(st));
  // affine normalisation on the host (one inversion); Z = 1
  if (std::is_same<C, G1>::value) {
    host::Fq x, y;
    if (!host::g1_to_affine(host::g1_from_device(h_res), &x, &y)) {
      std::memcpy(out_xyz, x.l, 48);
      std::memcpy(out_xyz + 6, y.l, 48);
      std::memcpy(out_xyz + 12, host::kOne, 48);
    }
  } else {
    host::Fq2 x, y;
    if (!host::g2_to_affine(host::g2_from_device(h_res), &x, &y)) {
      std::memcpy(out_xyz, &x, 96);
      std::memcpy(out_xyz + 12, &y, 96);
      std::memset(out_xyz + 24, 0, 96);
      std::memcpy(out_xyz + 24, host::kOne, 48);
    }
  }
}

template <class C>
void fixed_base_entry(Ctx& c, const uint64_t* scalars, uint64_t n, uint64_t* out_points, uint8_t* out_inf) {
  using Affine = typename C::Affine;
  B2Z_REQUIRE(n == 0 || (scalars && out_points && out_inf), B2Z_EINVAL, "fixed_base_mul: NULL argument");
  B2Z_REQUIRE(n < (1ull << 28), B2Z_ESIZE, "fixed_base_mul: more than 2^28 scalars in one call");
  if (n == 0) return;
  cudaStream_t st = c.stream;
  DevBuf<FrEl> ds(n);
  DevBuf<Affine> dp(n);
  DevBuf<uint32_t> dw((n + 31) / 32);
  B2Z_CUDA(cudaMemcpyAsync(ds.p, scalars, n * sizeof(FrEl), cudaMemcpyHostToDevice, st));
  if (std::is_same<C, G1>::value)
    g1_fixed_base_mul_device(&c, ds.p, reinterpret_cast<G1::Affine*>(dp.p), dw.p, (uint32_t)n, st);
  else
    g2_fixed_base_mul_device(&c, ds.p, reinterpret_cast<G2::Affine*>(dp.p), dw.p, (uint32_t)n, st);
  std::vector<uint32_t> words((n + 31) / 32);
  B2Z_CUDA(cudaMemcpyAsync(out_points, dp.p, n * sizeof(Affine), cudaMemcpyDeviceToHost, st));
  B2Z_CUDA(cudaMemcpyAsync(words.data(), dw.p, words.size() * 4, cudaMemcpyDeviceToHost, st));
  B2Z_CUDA(cudaStreamSynchronize(st));
  std::memcpy(out_inf, words.data(), (n + 7) / 8);
}

constexpr size_t kG1Bytes = sizeof(G1::Xyzz), kG2Bytes = sizeof(G2::Xyzz);
constexpr size_t kPartialBytes = 5 * kG1Bytes + kG2Bytes;   // A | sA | rB1 | L | H | B
constexpr size_t kPlaneSlotBytes = kMsmMaxPlanes * sizeof(G2::Xyzz);
static_assert(kPartialBytes == B2Z_PARTIAL_BYTES, "header constant out of sync");

// GPU part of a proof on this key (a whole key or one shard of it): leaves the XYZZ partial
// sums A, s*A, r*B1, L, H (G1) and B (G2) in partial_out (host memory).
// A proof in three steps that share the key's scratch (PkImpl): prove_begin launches everything that
// depends on z only, prove_quotient what needs the three coset evaluation vectors, prove_end waits and
// does the host epilogue.  The single-GPU prover runs them back to back; the sharded prover with a
// distributed witness map (b2z_groth16_shard_*) lets the caller exchange the coset evaluations between
// prove_begin and prove_quotient while the z-only accumulations are already running.
void prove_accums(Ctx& c, PkImpl& pk, cudaEvent_t gate = nullptr);
void prove_begin(Ctx& c, PkImpl& pk, const FrEl* d_z, const uint64_t r[4], const uint64_t s[4], bool with_accums = true) {
  ProofSum &A = pk.sums[SUM_A], &B1 = pk.sums[SUM_B1], &B = pk.sums[SUM_B], &L = pk.sums[SUM_L];
  // host-side scalars: r, s, -(r s) as canonical integers
  const FrEl r_m = Fr::reduce(fr_load_host(r)), s_m = Fr::reduce(fr_load_host(s));
  pk.r_c = Fr::from_mont(r_m);
  pk.s_c = Fr::from_mont(s_m);
  const FrEl neg_rs = Fr::from_mont(Fr::reduce(Fr::neg(Fr::reduce(Fr::mul(r_m, s_m)))));
  FrEl one_c = Fr::zero();
  one_c.l[0] = 1;
  const FrEl tail_h[5] = {one_c, pk.r_c, one_c, pk.s_c, neg_rs};      // A: {1, r}; B1, B: {1, s}; L: {-rs}
  B2Z_CUDA(cudaMemcpyAsync(pk.tail.p, tail_h, sizeof(tail_h), cudaMemcpyHostToDevice, A.stream));
  // this shard's variables of z as canonical integers
  if (pk.cyc_world == 0) {
    fr_from_mont_device(&c, d_z + pk.lo, pk.zc.p, pk.ma, A.stream);
  } else if (pk.ma) {
    fr_from_mont_cyclic_kernel<<<nblocks(pk.ma, 256), 256, 0, A.stream>>>(d_z, pk.zc.p, pk.ma, pk.cyc_rank,
                                                                          pk.cyc_world);
    B2Z_LAUNCHED(&c);
  }
  B2Z_CUDA(cudaEventRecord(pk.ev_z, A.stream));
  const FrEl* z_l = pk.zc.p + pk.l_skip;
  // ---- the four z-only sorts, concurrently
  msm_sort<G1>(&c, A.slot, pk.a_set, pk.zc.p, pk.ma, pk.tail.p + A.tail, A.stream);
  B2Z_CUDA(cudaStreamWaitEvent(B.stream, pk.ev_z, 0));
  msm_sort<G2>(&c, B.slot, pk.g2, pk.zc.p, pk.ma, pk.tail.p + B.tail, B.stream);
  B2Z_CUDA(cudaStreamWaitEvent(B1.stream, pk.ev_z, 0));
  msm_sort<G1>(&c, B1.slot, pk.b1_set, pk.zc.p, pk.ma, pk.tail.p + B1.tail, B1.stream);
  B2Z_CUDA(cudaStreamWaitEvent(L.stream, pk.ev_z, 0));
  msm_sort<G1>(&c, L.slot, pk.l_set, z_l, pk.ml, pk.tail.p + L.tail, L.stream);
  B2Z_CUDA(cudaEventRecord(L.sorted, L.stream));
  if (with_accums) prove_accums(c, pk);
}

// gate: fired when the witness map's transforms are done.  An accumulation kernel fills every SM for its whole
// duration (the G2 one takes all registers), so a transform queued beside it only runs in the gaps BETWEEN the
// accumulations and the H sum then waits for it with an idle GPU (8.7 of 100 ms at 2^22 before this gate).  The light
// phase -- sorts (latency / atomics bound) next to row evaluation and transforms (integer-pipe bound) -- overlaps
// well instead, and the accumulations then run back to back with the H sort hidden under them.
void prove_accums(Ctx& c, PkImpl& pk, cudaEvent_t gate) {
  ProofSum &A = pk.sums[SUM_A], &B1 = pk.sums[SUM_B1], &B = pk.sums[SUM_B], &L = pk.sums[SUM_L];
  // ---- accumulations chained by events (order below).  Each accumulation kernel is sized to fill the GPU by
  // itself; the G2 one (255 registers) leaves room for nothing, a G1 one leaves room on every SM for sort /
  // transform / tail blocks (the tail kernels are register-capped for exactly that), so tails overlap the next sums.
  // Every reduction stops at its bit-plane sums; the serial Horner pass over them, s*A and r*B1 are done
  // by the HOST (prove_end) while the GPU is still busy with L and H.  (With the scalar multiplications
  // on the GPU -- 1.5 ms each even with lane-cooperative arithmetic -- every order tried put one of them
  // on the critical path: 7.65-8.3 ms per C2 proof.)
  // Chaining only pays when an accumulation fills the GPU (148 SMs x 256 threads x >= 8 references each): below
  // ~256 k point references a kernel is latency-bound with idle SM slots, and the chain would just add the
  // kernels' latencies (Fibonacci: 5 variables; an eighth of the 16x16 matrix circuit) -- those run concurrently.
  auto big = [](uint64_t n, uint32_t windows) { return n * windows >= (1u << 18); };
  const bool chain = big(pk.g2.n, pk.g2.windows) || big(pk.a_set.n, pk.a_set.windows);
  auto after = [chain](const ProofSum& prev) { return chain ? prev.accum : nullptr; };
  // Order A -> B1 -> B (G2) -> L (-> H).  Two G1 sums open the chain because a G1 accumulation leaves a quarter of
  // every SM's registers free: the sorts of the other z-only MSMs (atomics-bound, starved while the transforms ran)
  // finish BESIDE them instead of in front of the G2 accumulation, which takes every register of every SM.  The
  // streams' priorities (api.cu) make the sorts finish in the order their sums need them.
  if (gate) B2Z_CUDA(cudaStreamWaitEvent(A.stream, gate, 0));
  msm_finish<G1>(&c, A.slot, pk.a_set, A.result<G1>(), A.stream, nullptr, A.accum, &A.planes);
  B2Z_CUDA(cudaEventRecord(A.done, A.stream));
  if (!chain && gate) {
    B2Z_CUDA(cudaStreamWaitEvent(B1.stream, gate, 0));
    B2Z_CUDA(cudaStreamWaitEvent(B.stream, gate, 0));
  }
  msm_finish<G1>(&c, B1.slot, pk.b1_set, B1.result<G1>(), B1.stream, after(A), B1.accum, &B1.planes);
  B2Z_CUDA(cudaEventRecord(B1.done, B1.stream));
  if (chain) B2Z_CUDA(cudaStreamWaitEvent(B.stream, L.sorted, 0));     // nothing runs beside the G2 sum: L's sort first
  msm_finish<G2>(&c, B.slot, pk.g2, B.result<G2>(), B.stream, after(B1), B.accum, &B.planes);
  B2Z_CUDA(cudaEventRecord(B.done, B.stream));
  msm_finish<G1>(&c, L.slot, pk.l_set, L.result<G1>(), L.stream, after(B), L.accum, &L.planes);
  B2Z_CUDA(cudaEventRecord(L.done, L.stream));
}

// d_a, d_b, d_c: evaluations of the three QAP combinations on the coset g H (d_a is clobbered)
void prove_h_finish(Ctx& c, PkImpl& pk, cudaStream_t st = nullptr) {
  const bool chain = (uint64_t)pk.h.n * pk.h.windows >= (1u << 18);
  ProofSum& H = pk.sums[SUM_H];
  H.stream = st ? st : c.stream;
  msm_finish<G1>(&c, H.slot, pk.h, H.result<G1>(), H.stream, chain ? pk.sums[SUM_L].accum : nullptr, nullptr,
                 &H.planes);
}
void prove_quotient(Ctx& c, PkImpl& pk, FrEl* d_a, const FrEl* d_b, const FrEl* d_c, bool with_h_finish = true) {
  cudaStream_t st = c.stream;
  witness_map_quotient(&c, d_a, d_b, d_c, pk.log_n, /*natural_out=*/false, st);    // whole domain, every shard
  B2Z_CUDA(cudaEventRecord(pk.ev_wm, st));
  fr_from_mont_device(&c, d_a + pk.h_lo, pk.hc.p, pk.hn, st);
  msm_sort<G1>(&c, pk.sums[SUM_H].slot, pk.h, pk.hc.p, pk.hn, nullptr, st);
  if (with_h_finish) prove_h_finish(c, pk);
}

void prove_end(Ctx& c, PkImpl& pk, uint8_t* partial_out) {
  auto planes = [&](Sum k) { return static_cast<const uint32_t*>(pk.sums[k].planes.host); };
  auto g1_result = [&](Sum k) { return host::g1_planes_horner(planes(k), pk.sums[k].planes.nplanes, kMsmChunkLog); };
  // A, s*A, B1, r*B1 while the GPU works on L and H
  B2Z_CUDA(cudaEventSynchronize(pk.sums[SUM_A].done));
  const host::G1Xyzz A = g1_result(SUM_A);
  host::g1_to_device_layout(A, pk.h_out + 0 * kG1Bytes / 4);
  host::g1_to_device_layout(host::g1_mul_scalar(A, pk.s_c.l), pk.h_out + 1 * kG1Bytes / 4);
  B2Z_CUDA(cudaEventSynchronize(pk.sums[SUM_B1].done));
  host::g1_to_device_layout(host::g1_mul_scalar(g1_result(SUM_B1), pk.r_c.l), pk.h_out + 2 * kG1Bytes / 4);
  B2Z_CUDA(cudaEventSynchronize(pk.sums[SUM_B].done));
  host::g2_to_device_layout(host::g2_planes_horner(planes(SUM_B), pk.sums[SUM_B].planes.nplanes, kMsmChunkLog),
                            pk.h_out + 5 * kG1Bytes / 4);
  B2Z_CUDA(cudaEventSynchronize(pk.sums[SUM_L].done));
  host::g1_to_device_layout(g1_result(SUM_L), pk.h_out + 3 * kG1Bytes / 4);
  B2Z_CUDA(cudaStreamSynchronize(pk.sums[SUM_H].stream));
  host::g1_to_device_layout(g1_result(SUM_H), pk.h_out + 4 * kG1Bytes / 4);
  std::memcpy(partial_out, pk.h_out, kPartialBytes);
}

void prove_partial_device(Ctx& c, PkImpl& pk, FrEl* d_a, FrEl* d_b, FrEl* d_c, const FrEl* d_z, const uint64_t r[4],
                          const uint64_t s[4], uint8_t* partial_out) {
  // issue order: everything light first (sorts, witness map, H sort), then the GPU-filling accumulations
  prove_begin(c, pk, d_z, r, s, /*with_accums=*/false);
  witness_map_transform3(&c, d_a, d_b, d_c, pk.log_n, c.stream);
  prove_quotient(c, pk, d_a, d_b, d_c, /*with_h_finish=*/false);
  // small domains: the transforms run in 128-thread CTAs that fit on an SM beside a G1 accumulation and fill its
  // idle issue slots (the accumulations are latency-bound there), so no gate
  prove_accums(c, pk, pk.log_n >= 19 ? pk.ev_wm : nullptr);
  prove_h_finish(c, pk);
  prove_end(c, pk, partial_out);
}

// Host epilogue: sum the partials of all shards, normalise, serialise (host_fq.hpp).
void combine_partials(const uint8_t* partials, uint32_t world, uint8_t proof_out[192]) {
  host::G1Xyzz A, C;
  host::G2Xyzz B;
  std::memset(&A, 0, sizeof(A));
  std::memset(&C, 0, sizeof(C));
  std::memset(&B, 0, sizeof(B));
  for (uint32_t k = 0; k < world; k++) {
    uint32_t w[kPartialBytes / 4];
    std::memcpy(w, partials + (size_t)k * kPartialBytes, kPartialBytes);
    A = host::g1_add(A, host::g1_from_device(w));
    for (int j = 1; j < 5; j++) C = host::g1_add(C, host::g1_from_device(w + j * kG1Bytes / 4));   // sA + rB1 + L + H
    B = host::g2_add(B, host::g2_from_device(w + 5 * kG1Bytes / 4));
  }
  host::g1_serialize(proof_out, A);
  host::g2_serialize(proof_out + 48, B);
  host::g1_serialize(proof_out + 144, C);
}

void prove_device(Ctx& c, PkImpl& pk, FrEl* d_a, FrEl* d_b, FrEl* d_c, const FrEl* d_z, const uint64_t r[4],
                  const uint64_t s[4], uint8_t proof_out[192]) {
  B2Z_REQUIRE(pk.with_vk && pk.ma == pk.m && pk.hn == (1u << pk.log_n), B2Z_EINVAL,
              "b2z_groth16_prove needs a whole key; use b2z_groth16_prove_partial + b2z_groth16_combine on shards");
  uint8_t partial[kPartialBytes];
  prove_partial_device(c, pk, d_a, d_b, d_c, d_z, r, s, partial);
  combine_partials(partial, 1, proof_out);
}

}  // namespace
}  // namespace b2z

using namespace b2z;

struct b2z_pk {
  PkImpl impl;
};

namespace b2z {
// the key's scratch is per-proof state: only the context that uploaded it may prove on it
PkImpl& pk_of(Ctx& c, const b2z_pk* pk, const char* who) {
  if (pk == nullptr) throw StatusError{B2Z_EINVAL, std::string(who) + ": key is NULL"};
  PkImpl& P = const_cast<b2z_pk*>(pk)->impl;
  if (P.owner != &c)
    throw StatusError{B2Z_EINVAL, std::string(who) + ": this b2z_pk was uploaded through another b2z_ctx (a key handle "
                                                     "belongs to one context; upload one copy per context)"};
  return P;
}
bool pk_matches(const b2z_pk* pk, uint32_t log_n, uint64_t m, uint64_t l) {
  return pk->impl.log_n == log_n && pk->impl.m == m && pk->impl.l == l;
}
void prove_on_device_buffers(Ctx& c, const b2z_pk* pk, FrEl* d_a, FrEl* d_b, FrEl* d_c, const FrEl* d_z,
                             const uint64_t r[4], const uint64_t s[4], uint8_t proof_out[192]) {
  prove_device(c, pk_of(c, pk, "b2z_groth16_prove"), d_a, d_b, d_c, d_z, r, s, proof_out);
}
void prove_partial_on_device_buffers(Ctx& c, const b2z_pk* pk, FrEl* d_a, FrEl* d_b, FrEl* d_c, const FrEl* d_z,
                                     const uint64_t r[4], const uint64_t s[4], uint8_t* partial_out) {
  prove_partial_device(c, pk_of(c, pk, "b2z_groth16_prove_partial"), d_a, d_b, d_c, d_z, r, s, partial_out);
}
void prove_begin_on(Ctx& c, const b2z_pk* pk, const FrEl* d_z, const uint64_t r[4], const uint64_t s[4]) {
  prove_begin(c, pk_of(c, pk, "b2z_groth16_shard_begin"), d_z, r, s);
}
// ---- pieces of a proof for the tile-sharded (distributed witness map) prover in r1cs.cu
void prove_begin_sorts_on(Ctx& c, const b2z_pk* pk, const FrEl* d_z, const uint64_t r[4], const uint64_t s[4]) {
  prove_begin(c, pk_of(c, pk, "b2z_dist_prove"), d_z, r, s, /*with_accums=*/false);
}
uint32_t pk_h_chunk(const b2z_pk* pk, uint32_t* h_lo) {
  if (h_lo) *h_lo = pk->impl.h_lo;
  return pk->impl.hn;
}
// d_h: this shard's hn coefficients of h (bit-reversed positions [h_lo, h_lo + hn)), canonical Montgomery form
void prove_dist_h_sort_on(Ctx& c, const b2z_pk* pk, const FrEl* d_h, cudaStream_t st) {
  PkImpl& P = pk_of(c, pk, "b2z_dist_prove");
  fr_from_mont_device(&c, d_h, P.hc.p, P.hn, st);
  msm_sort<G1>(&c, P.sums[SUM_H].slot, P.h, P.hc.p, P.hn, nullptr, st);
}
// all five accumulations, chained: the first once `wm_done` has fired (the witness map's transform kernels need the
// SMs the accumulations would fill), H on `h_st` -- the stream its sort was queued on, which therefore hides under
// the other accumulations; then the host epilogue
void prove_dist_finish_on(Ctx& c, const b2z_pk* pk, cudaEvent_t wm_done, cudaStream_t h_st, uint8_t* partial_out) {
  PkImpl& P = pk_of(c, pk, "b2z_dist_prove");
  prove_accums(c, P, wm_done);                            // the G2 accumulation opens the chain
  prove_h_finish(c, P, h_st);
  prove_end(c, P, partial_out);
}
void combine_partials_host(const uint8_t* partials, uint32_t world, uint8_t proof_out[192]) {
  combine_partials(partials, world, proof_out);
}
void pk_bind_assignment_flag(const b2z_pk* pk, bool* flag) { const_cast<b2z_pk*>(pk)->impl.assignment_flag = flag; }
void prove_finish_on(Ctx& c, const b2z_pk* pk, FrEl* d_a, const FrEl* d_b, const FrEl* d_c, uint8_t* partial_out) {
  PkImpl& P = pk_of(c, pk, "b2z_groth16_shard_finish");
  if (P.assignment_flag != nullptr) {
    *P.assignment_flag = false;
    P.assignment_flag = nullptr;
  }
  prove_quotient(c, P, d_a, d_b, d_c);
  prove_end(c, P, partial_out);
}
}  // namespace b2z

extern "C" {

b2z_status b2z_msm_g1(b2z_ctx* ctx, const uint64_t* bases, const uint8_t* inf_bitmap, const uint64_t* scalars,
                      uint64_t n, uint64_t out_xyz[18]) {
  return guarded(ctx, [&](Ctx& c) { msm_entry<G1>(c, bases, inf_bitmap, scalars, n, out_xyz); });
}

b2z_status b2z_msm_g2(b2z_ctx* ctx, const uint64_t* bases, const uint8_t* inf_bitmap, const uint64_t* scalars,
                      uint64_t n, uint64_t out_xyz[36]) {
  return guarded(ctx, [&](Ctx& c) { msm_entry<G2>(c, bases, inf_bitmap, scalars, n, out_xyz); });
}

b2z_status b2z_fixed_base_mul_g1(b2z_ctx* ctx, const uint64_t* scalars, uint64_t n, uint64_t* out_points,
                                 uint8_t* out_inf) {
  return guarded(ctx, [&](Ctx& c) { fixed_base_entry<G1>(c, scalars, n, out_points, out_inf); });
}

b2z_status b2z_fixed_base_mul_g2(b2z_ctx* ctx, const uint64_t* scalars, uint64_t n, uint64_t* out_points,
                                 uint8_t* out_inf) {
  return guarded(ctx, [&](Ctx& c) { fixed_base_entry<G2>(c, scalars, n, out_points, out_inf); });
}

// from / to / den: contiguous slice of the variables AND of the h positions.  cyc_world > 0: the h positions still
// follow from / to / den, the variables are the block-cyclic subset of rank cyc_rank of cyc_world.
static b2z_status pk_upload_impl(b2z_ctx* ctx, const b2z_pk_desc* d, uint32_t from, uint32_t to, uint32_t den,
                                 uint32_t cyc_rank, uint32_t cyc_world, b2z_pk** out) {
  if (out) *out = nullptr;
  return guarded(ctx, [&](Ctx& c) {
    B2Z_REQUIRE(d != nullptr && out != nullptr, B2Z_EINVAL, "b2z_pk_upload: NULL argument");
    B2Z_REQUIRE(den >= 1 && from <= to && to <= den, B2Z_EINVAL, "b2z_pk_upload_slice: need from <= to <= den");
    B2Z_REQUIRE(d->log_domain <= 32, B2Z_ESIZE, "b2z_pk_upload: domain larger than 2^32");
    B2Z_REQUIRE(d->log_domain <= 26, B2Z_ENOMEM, "b2z_pk_upload: domain does not fit this build's single-GPU plan");
    B2Z_REQUIRE(d->num_instance >= 1 && d->num_variables >= d->num_instance, B2Z_EINVAL,
                "b2z_pk_upload: need 1 <= num_instance <= num_variables");
    const uint64_t m = d->num_variables, l = d->num_instance, n = 1ull << d->log_domain;
    B2Z_REQUIRE(m < (1ull << 26), B2Z_ESIZE, "b2z_pk_upload: too many variables");
    B2Z_REQUIRE(d->a_query && d->b_g1_query && d->b_g2_query && (n == 1 || d->h_query) && (m == l || d->l_query) &&
                    d->alpha_g1 && d->beta_g1 && d->delta_g1 && d->beta_g2 && d->delta_g2,
                B2Z_EINVAL, "b2z_pk_upload: NULL query array");
    std::unique_ptr<b2z_pk> pk(new b2z_pk());
    PkImpl& P = pk->impl;
    P.owner = &c;
    P.log_n = d->log_domain;
    P.m = m;
    P.l = l;
    // the variables of this shard, in local order
    if (cyc_world > 0 && l > kCycBlock) cyc_world = 0;   // the instance variables must sit in block 0
    uint64_t lo = m * from / den, hi = m * to / den;
    std::vector<uint32_t> ids;                           // cyclic mode only
    if (cyc_world > 0) {
      for (uint64_t b = cyc_rank; b * kCycBlock < m; b += cyc_world)
        for (uint64_t i = b * kCycBlock; i < (b + 1) * kCycBlock && i < m; i++) ids.push_back((uint32_t)i);
      P.cyc_world = cyc_world; P.cyc_rank = cyc_rank;
      P.lo = 0; P.ma = (uint32_t)ids.size();
      P.l_skip = cyc_rank == 0 ? (uint32_t)(l < P.ma ? l : P.ma) : 0;
      lo = 0; hi = P.ma;
    } else {
      const uint64_t l_lo = lo > l ? lo : l;             // first witness variable in the slice
      P.lo = (uint32_t)lo; P.ma = (uint32_t)(hi - lo);
      P.l_skip = (uint32_t)((l_lo < hi ? l_lo : hi) - lo);
    }
    P.ml = P.ma - P.l_skip;
    const uint64_t h_lo = n * from / den, h_hi = n * to / den;
    P.h_lo = (uint32_t)h_lo; P.hn = (uint32_t)(h_hi - h_lo);
    P.with_vk = from == 0 ? 1u : 0u;
    cudaStream_t st = c.stream;
    size_t free_b = 0, total_b = 0;
    B2Z_CUDA(cudaMemGetInfo(&free_b, &total_b));
    const bool pre = pk_precompute_bytes(d) / den * (to - from) < free_b / 2;
    // `count` points of a query, starting at local variable `skip` of this shard, as one contiguous host array
    // (query index = variable index - shift) + identity bits; contiguous shards point straight into the caller's array
    struct Picked {
      const uint64_t* pts = nullptr;
      const uint8_t* inf = nullptr;
      std::vector<uint64_t> own_pts;
      std::vector<uint8_t> own_inf;
    };
    auto pick = [&](Picked& out, const uint64_t* query, const uint8_t* inf, uint32_t skip, uint32_t count, uint64_t shift,
                    uint32_t limbs) {
      if (count == 0 || query == nullptr) return;
      auto var = [&](uint32_t j) { return cyc_world > 0 ? (uint64_t)ids[j] : lo + j; };
      if (cyc_world == 0) {
        out.pts = query + (size_t)limbs * (var(skip) - shift);
      } else {
        out.own_pts.resize((size_t)limbs * count);
        for (uint32_t j = 0; j < count;) {               // copy block by block
          const uint64_t q = var(skip + j) - shift;
          uint32_t run = 1;
          while (j + run < count && var(skip + j + run) - shift == q + run) run++;
          std::memcpy(&out.own_pts[(size_t)limbs * j], query + (size_t)limbs * q, (size_t)limbs * 8 * run);
          j += run;
        }
        out.pts = out.own_pts.data();
      }
      if (inf != nullptr) {
        out.own_inf.assign((count + 7) / 8 + 1, 0);
        for (uint32_t j = 0; j < count; j++) {
          const uint64_t q = var(skip + j) - shift;
          if ((inf[q >> 3] >> (q & 7)) & 1) out.own_inf[j >> 3] |= (uint8_t)(1u << (j & 7));
        }
        out.inf = out.own_inf.data();
      }
    };
    // one G1 set = the picked query points, then up to two vk points (shard 0 only)
    auto build_g1 = [&](MsmBases<G1>& out, const uint64_t* query, const uint8_t* inf, uint32_t skip, uint32_t count,
                        uint64_t shift, const uint64_t* extra0, const uint64_t* extra1) {
      const uint32_t extras = P.with_vk ? ((extra0 ? 1 : 0) + (extra1 ? 1 : 0)) : 0;
      const uint32_t total = count + extras;
      DevBuf<G1::Affine> dpts(total ? total : 1);
      std::vector<uint32_t> words((total + 31) / 32 + 1, 0u);
      Picked pk_pts;
      pick(pk_pts, query, inf, skip, count, shift, 12);
      stage_points<G1::Affine>(dpts.p, words, 0, pk_pts.pts, pk_pts.inf, count, st);
      uint64_t at = count;
      if (P.with_vk && extra0) stage_points<G1::Affine>(dpts.p, words, at++, extra0, nullptr, 1, st);
      if (P.with_vk && extra1) stage_points<G1::Affine>(dpts.p, words, at++, extra1, nullptr, 1, st);
      DevBuf<uint32_t> dinf(words.size());
      B2Z_CUDA(cudaMemcpyAsync(dinf.p, words.data(), words.size() * 4, cudaMemcpyHostToDevice, st));
      msm_bases_build<G1>(&c, out, dpts.p, dinf.p, total, pre, 0, st);
      B2Z_CUDA(cudaStreamSynchronize(st));
    };
    build_g1(P.a_set, d->a_query, d->a_inf, 0, P.ma, 0, d->alpha_g1, d->delta_g1);
    build_g1(P.b1_set, d->b_g1_query, d->b_g1_inf, 0, P.ma, 0, d->beta_g1, d->delta_g1);
    build_g1(P.l_set, d->l_query, d->l_inf, P.l_skip, P.ml, l, d->delta_g1, nullptr);
    {
      // G2: [b2 | beta_2 delta_2]
      const uint32_t n2 = P.ma + (P.with_vk ? 2 : 0);
      DevBuf<G2::Affine> dpts(n2 ? n2 : 1);
      std::vector<uint32_t> words((n2 + 31) / 32 + 1, 0u);
      Picked g2_pts;
      pick(g2_pts, d->b_g2_query, d->b_g2_inf, 0, P.ma, 0, 24);
      stage_points<G2::Affine>(dpts.p, words, 0, g2_pts.pts, g2_pts.inf, P.ma, st);
      if (P.with_vk) {
        stage_points<G2::Affine>(dpts.p, words, P.ma, d->beta_g2, nullptr, 1, st);
        stage_points<G2::Affine>(dpts.p, words, (uint64_t)P.ma + 1, d->delta_g2, nullptr, 1, st);
      }
      DevBuf<uint32_t> dinf(words.size());
      B2Z_CUDA(cudaMemcpyAsync(dinf.p, words.data(), words.size() * 4, cudaMemcpyHostToDevice, st));
      msm_bases_build<G2>(&c, P.g2, dpts.p, dinf.p, n2, pre, 0, st);
      B2Z_CUDA(cudaStreamSynchronize(st));
    }
    {
      // h_query in bit-reversed order, padded to n with a flagged identity; keep positions [h_lo, h_hi)
      DevBuf<G1::Affine> src(n), dst(n);
      DevBuf<uint32_t> src_inf, flags(n), words((P.hn + 31) / 32 + 1);
      if (n > 1) B2Z_CUDA(cudaMemcpyAsync(src.p, d->h_query, (n - 1) * sizeof(G1::Affine), cudaMemcpyHostToDevice, st));
      std::vector<uint32_t> hw;
      if (d->h_inf != nullptr && n > 1) {
        hw.assign((n + 31) / 32, 0u);
        std::memcpy(hw.data(), d->h_inf, (n - 1 + 7) / 8);
        src_inf.alloc(hw.size());
        B2Z_CUDA(cudaMemcpyAsync(src_inf.p, hw.data(), hw.size() * 4, cudaMemcpyHostToDevice, st));
      }
      permute_bitrev_g1_kernel<<<nblocks(n, 256), 256, 0, st>>>(src.p, src_inf.p, (uint32_t)(n - 1), P.log_n, dst.p,
                                                                flags.p);
      B2Z_LAUNCHED(&c);
      pack_flags_device(&c, flags.p + h_lo, P.hn, words.p, st);
      msm_bases_build<G1>(&c, P.h, dst.p + h_lo, words.p, P.hn, pre, 0, st);
      B2Z_CUDA(cudaStreamSynchronize(st));
    }
    P.ea.alloc(n); P.eb.alloc(n); P.ec.alloc(n); P.hc.alloc(P.hn ? P.hn : 1);
    P.z.alloc(m); P.zc.alloc(P.ma ? P.ma : 1); P.tail.alloc(5);
    P.g1_out.alloc(SUM_B); P.g2_out.alloc(1);
    B2Z_CUDA(cudaMallocHost(&P.h_out, kPartialBytes));
    B2Z_CUDA(cudaMallocHost(&P.h_planes, SUM_COUNT * kPlaneSlotBytes));
    auto new_event = [](cudaEvent_t* e) { B2Z_CUDA(cudaEventCreateWithFlags(e, cudaEventDisableTiming)); };
    auto init = [&](Sum k, int slot, cudaStream_t stream, uint32_t tail, void* d_result) {
      ProofSum& S = P.sums[k];
      S.slot = slot;
      S.stream = stream;
      S.tail = tail;
      S.d_result = d_result;
      S.planes.host = P.h_planes + (size_t)k * kPlaneSlotBytes / 4;
      if (k != SUM_H) {
        new_event(&S.accum);
        new_event(&S.done);
      }
    };
    // arena slot, stream (H: the one prove_h_finish names), offset of the tail scalars in {1, r, 1, s, -rs}, result
    init(SUM_A, 1, c.aux[0], 0, P.g1_out.p + SUM_A);
    init(SUM_B1, 3, c.aux[2], 2, P.g1_out.p + SUM_B1);
    init(SUM_L, 4, c.aux[3], 4, P.g1_out.p + SUM_L);
    init(SUM_H, 0, c.stream, 0, P.g1_out.p + SUM_H);
    init(SUM_B, 2, c.aux[1], 2, P.g2_out.p);
    new_event(&P.sums[SUM_L].sorted);
    new_event(&P.ev_z);
    new_event(&P.ev_wm);
    *out = pk.release();
  });
}

b2z_status b2z_pk_upload_slice(b2z_ctx* ctx, const b2z_pk_desc* d, uint32_t from, uint32_t to, uint32_t den,
                               b2z_pk** out) {
  return pk_upload_impl(ctx, d, from, to, den, 0, 0, out);
}

b2z_status b2z_pk_upload_shard(b2z_ctx* ctx, const b2z_pk_desc* d, uint32_t rank, uint32_t world, b2z_pk** out) {
  if (world < 1 || rank >= world) {
    if (out) *out = nullptr;
    return guarded(ctx, [&](Ctx&) { B2Z_REQUIRE(false, B2Z_EINVAL, "b2z_pk_upload_shard: need rank < world"); });
  }
  // variables block-cyclic over the ranks (balanced for any witness), h positions in contiguous chunks
  return pk_upload_impl(ctx, d, rank, rank + 1, world, rank, world > 1 ? world : 0, out);
}

b2z_status b2z_pk_upload(b2z_ctx* ctx, const b2z_pk_desc* d, b2z_pk** out) {
  return b2z_pk_upload_slice(ctx, d, 0, 1, 1, out);
}

b2z_status b2z_groth16_prove_partial(b2z_ctx* ctx, const b2z_pk* pk_c, const uint64_t* a_evals, const uint64_t* b_evals,
                                     const uint64_t* c_evals, const uint64_t* z, const uint64_t r[4],
                                     const uint64_t s[4], uint8_t* partial_out) {
  return guarded(ctx, [&](Ctx& c) {
    B2Z_REQUIRE(pk_c && a_evals && b_evals && c_evals && z && r && s && partial_out, B2Z_EINVAL,
                "b2z_groth16_prove_partial: NULL argument");
    PkImpl& P = pk_of(c, pk_c, "b2z_groth16_prove_partial");
    const size_t n = (size_t)1 << P.log_n;
    B2Z_CUDA(cudaMemcpyAsync(P.z.p, z, P.m * sizeof(FrEl), cudaMemcpyHostToDevice, c.aux[0]));
    B2Z_CUDA(cudaMemcpyAsync(P.ea.p, a_evals, n * sizeof(FrEl), cudaMemcpyHostToDevice, c.stream));
    B2Z_CUDA(cudaMemcpyAsync(P.eb.p, b_evals, n * sizeof(FrEl), cudaMemcpyHostToDevice, c.stream));
    B2Z_CUDA(cudaMemcpyAsync(P.ec.p, c_evals, n * sizeof(FrEl), cudaMemcpyHostToDevice, c.stream));
    prove_partial_device(c, P, P.ea.p, P.eb.p, P.ec.p, P.z.p, r, s, partial_out);
  });
}

b2z_status b2z_groth16_combine(const uint8_t* partials, uint32_t world, uint8_t proof_out[192]) {
  if (partials == nullptr || proof_out == nullptr || world == 0) return B2Z_EINVAL;
  combine_partials(partials, world, proof_out);
  return B2Z_OK;
}

void b2z_pk_free(b2z_ctx* ctx, b2z_pk* pk) {
  if (pk == nullptr) return;
  if (ctx != nullptr) {
    std::lock_guard<std::mutex> lock(ctx->impl.mu);
    cudaSetDevice(ctx->impl.device);
    cudaDeviceSynchronize();
    delete pk;
  } else {
    delete pk;
  }
}

b2z_status b2z_groth16_prove(b2z_ctx* ctx, const b2z_pk* pk_c, const uint64_t* a_evals, const uint64_t* b_evals,
                             const uint64_t* c_evals, const uint64_t* z, const uint64_t r[4], const uint64_t s[4],
                             uint8_t proof_out[192]) {
  return guarded(ctx, [&](Ctx& c) {
    B2Z_REQUIRE(pk_c && a_evals && b_evals && c_evals && z && r && s && proof_out, B2Z_EINVAL,
                "b2z_groth16_prove: NULL argument");
    PkImpl& P = pk_of(c, pk_c, "b2z_groth16_prove");
    const size_t n = (size_t)1 << P.log_n;
    B2Z_CUDA(cudaMemcpyAsync(P.z.p, z, P.m * sizeof(FrEl), cudaMemcpyHostToDevice, c.aux[0]));
    B2Z_CUDA(cudaMemcpyAsync(P.ea.p, a_evals, n * sizeof(FrEl), cudaMemcpyHostToDevice, c.stream));
    B2Z_CUDA(cudaMemcpyAsync(P.eb.p, b_evals, n * sizeof(FrEl), cudaMemcpyHostToDevice, c.stream));
    B2Z_CUDA(cudaMemcpyAsync(P.ec.p, c_evals, n * sizeof(FrEl), cudaMemcpyHostToDevice, c.stream));
    prove_device(c, P, P.ea.p, P.eb.p, P.ec.p, P.z.p, r, s, proof_out);
  });
}

b2z_status b2z_groth16_prove_device(b2z_ctx* ctx, const b2z_pk* pk_c, uint64_t* d_a, uint64_t* d_b, uint64_t* d_c,
                                    const uint64_t* d_z, const uint64_t r[4], const uint64_t s[4],
                                    uint8_t proof_out[192]) {
  return guarded(ctx, [&](Ctx& c) {
    B2Z_REQUIRE(pk_c && d_a && d_b && d_c && d_z && r && s && proof_out, B2Z_EINVAL,
                "b2z_groth16_prove_device: NULL argument");
    PkImpl& P = pk_of(c, pk_c, "b2z_groth16_prove_device");
    // The caller's buffers must be complete, or produced on the legacy default stream (what a torch / plain-CUDA
    // caller uses): the library's non-blocking streams are ordered after it by an event -- no device-wide
    // synchronisation, which would serialise every context that shares this GPU.
    B2Z_CUDA(cudaEventRecord(P.ev_z, cudaStreamLegacy));
    B2Z_CUDA(cudaStreamWaitEvent(c.stream, P.ev_z, 0));
    B2Z_CUDA(cudaStreamWaitEvent(c.aux[0], P.ev_z, 0));
    prove_device(c, P, reinterpret_cast<FrEl*>(d_a), reinterpret_cast<FrEl*>(d_b), reinterpret_cast<FrEl*>(d_c),
                 reinterpret_cast<const FrEl*>(d_z), r, s, proof_out);
  });
}

}  // extern "C"
