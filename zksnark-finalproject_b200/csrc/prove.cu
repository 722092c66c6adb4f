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

constexpr size_t kG1Bytes = sizeof(G1::Xyzz), kG2Bytes = sizeof(G2::Xyzz);
constexpr size_t kPartialBytes = 5 * kG1Bytes + kG2Bytes;   // A | sA | rB1 | L | H | B
constexpr size_t kPlaneSlotBytes = kMsmMaxPlanes * sizeof(G2::Xyzz);
static_assert(kPartialBytes == B2Z_PARTIAL_BYTES, "header constant out of sync");

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

// per-proof scratch, the proof's sums (arena slot, stream, tail offset, result) and events; after the shard fields
void pk_alloc_scratch(Ctx& c, PkImpl& P) {
  const uint64_t n = 1ull << P.log_n;
  P.ea.alloc(n); P.eb.alloc(n); P.ec.alloc(n); P.hc.alloc(P.hn ? P.hn : 1);
  P.z.alloc(P.m); P.zc.alloc(P.ma ? P.ma : 1); P.tail.alloc(5);
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
  // arena slot, stream (H: set by proof_h_sort), offset of the tail scalars in {1, r, 1, s, -rs}, result
  init(SUM_A, 1, c.aux[0], 0, P.g1_out.p + SUM_A);
  init(SUM_B1, 3, c.aux[2], 2, P.g1_out.p + SUM_B1);
  init(SUM_L, 4, c.aux[3], 4, P.g1_out.p + SUM_L);
  init(SUM_H, 0, nullptr, 0, P.g1_out.p + SUM_H);
  init(SUM_B, 2, c.aux[1], 2, P.g2_out.p);
  new_event(&P.sums[SUM_L].sorted);
  new_event(&P.ev_z);
  new_event(&P.ev_wm);
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


// the host-side a/b/c evaluations and assignment of b2z_groth16_prove[_partial] into the key's scratch: z on the
// stream that prepares the MSM scalars, the evaluations on the main stream
void stage_host_inputs(Ctx& c, PkImpl& P, const uint64_t* a, const uint64_t* b, const uint64_t* cc, const uint64_t* z) {
  const size_t n = (size_t)1 << P.log_n;
  B2Z_CUDA(cudaMemcpyAsync(P.z.p, z, P.m * sizeof(FrEl), cudaMemcpyHostToDevice, c.aux[0]));
  B2Z_CUDA(cudaMemcpyAsync(P.ea.p, a, n * sizeof(FrEl), cudaMemcpyHostToDevice, c.stream));
  B2Z_CUDA(cudaMemcpyAsync(P.eb.p, b, n * sizeof(FrEl), cudaMemcpyHostToDevice, c.stream));
  B2Z_CUDA(cudaMemcpyAsync(P.ec.p, cc, n * sizeof(FrEl), cudaMemcpyHostToDevice, c.stream));
}

}  // namespace

// ---------------------------------------------------------------------------
// The five phases of a proof (prove_internal.hpp).  prove_partial_device and b2z_dist_prove issue the light work
// first -- scalar prep, the sorts, the witness map, the H sort -- and then the GPU-filling accumulations back to back;
// b2z_groth16_shard_begin starts the z-only accumulations at once, while the caller exchanges the coset evaluations
// that b2z_groth16_shard_finish takes.
// ---------------------------------------------------------------------------
void proof_begin(Ctx& c, PkImpl& pk, const FrEl* d_z, const uint64_t r[4], const uint64_t s[4]) {
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
}

void proof_h_sort(Ctx& c, PkImpl& pk, const FrEl* d_h, cudaStream_t st) {
  ProofSum& H = pk.sums[SUM_H];
  H.stream = st;
  fr_from_mont_device(&c, d_h, pk.hc.p, pk.hn, st);
  msm_sort<G1>(&c, H.slot, pk.h, pk.hc.p, pk.hn, nullptr, st);
}

// gate: fired when the witness map's transforms are done.  An accumulation kernel fills every SM for its whole
// duration (the G2 one takes all registers), so a transform queued beside it only runs in the gaps BETWEEN the
// accumulations and the H sum then waits for it with an idle GPU (8.7 of 100 ms at 2^22 before this gate).  The light
// phase -- sorts (latency / atomics bound) next to row evaluation and transforms (integer-pipe bound) -- overlaps
// well instead, and the accumulations then run back to back with the H sort hidden under them.
void proof_accums(Ctx& c, PkImpl& pk, cudaEvent_t gate) {
  ProofSum &A = pk.sums[SUM_A], &B1 = pk.sums[SUM_B1], &B = pk.sums[SUM_B], &L = pk.sums[SUM_L];
  // ---- accumulations chained by events (order below).  Each accumulation kernel is sized to fill the GPU by
  // itself; the G2 one (255 registers) leaves room for nothing, a G1 one leaves room on every SM for sort /
  // transform / tail blocks (the tail kernels are register-capped for exactly that), so tails overlap the next sums.
  // Every reduction stops at its bit-plane sums; the serial Horner pass over them, s*A and r*B1 are done
  // by the HOST (proof_end) while the GPU is still busy with L and H.  (With the scalar multiplications
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

void proof_h_finish(Ctx& c, PkImpl& pk) {
  const bool chain = (uint64_t)pk.h.n * pk.h.windows >= (1u << 18);
  ProofSum& H = pk.sums[SUM_H];
  msm_finish<G1>(&c, H.slot, pk.h, H.result<G1>(), H.stream, chain ? pk.sums[SUM_L].accum : nullptr, nullptr,
                 &H.planes);
}

void proof_end(Ctx& c, PkImpl& pk, uint8_t* partial_out) {
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
  proof_begin(c, pk, d_z, r, s);
  witness_map_transform3(&c, d_a, d_b, d_c, pk.log_n, c.stream);
  witness_map_quotient(&c, d_a, d_b, d_c, pk.log_n, /*natural_out=*/false, c.stream);    // whole domain, every shard
  B2Z_CUDA(cudaEventRecord(pk.ev_wm, c.stream));
  proof_h_sort(c, pk, d_a + pk.h_lo, c.stream);
  // small domains: the transforms run in 128-thread CTAs that fit on an SM beside a G1 accumulation and fill its
  // idle issue slots (the accumulations are latency-bound there), so no gate
  proof_accums(c, pk, pk.log_n >= 19 ? pk.ev_wm : nullptr);
  proof_h_finish(c, pk);
  proof_end(c, pk, partial_out);
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
  B2Z_REQUIRE(pk.whole(), B2Z_EINVAL,
              "b2z_groth16_prove needs a whole key; use b2z_groth16_prove_partial + b2z_groth16_combine on shards");
  uint8_t partial[kPartialBytes];
  prove_partial_device(c, pk, d_a, d_b, d_c, d_z, r, s, partial);
  combine_partials(partial, 1, proof_out);
}
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
// `num` / `den` of the key's precomputed window copies fit in half the free device memory
bool pk_precompute_fits_slice(uint32_t log_n, uint64_t m, uint64_t l, uint32_t num, uint32_t den) {
  auto cost = [](uint64_t n, size_t pt) {
    if (n == 0) return (size_t)0;
    const uint32_t c = msm_pick_c(n, true);
    return (size_t)n * pt * msm_windows(c);
  };
  const uint64_t n = 1ull << log_n;
  const size_t bytes = 2 * cost(m + 2, 96) + cost(m - l + 1, 96) + cost(m + 2, 192) + cost(n, 96);
  size_t free_b = 0, total_b = 0;
  B2Z_CUDA(cudaMemGetInfo(&free_b, &total_b));
  return bytes / den * num < free_b / 2;
}
b2z_pk* pk_from_device_sets(Ctx& c, const PkShard& shard, const PkDeviceSets& S, bool pre) {
  std::unique_ptr<b2z_pk> pk(new b2z_pk());
  PkImpl& P = pk->impl;
  P.owner = &c;
  static_cast<PkShard&>(P) = shard;
  const uint32_t vk_terms = P.with_vk ? 2 : 0;   // alpha/beta/delta (a, b1, b2) and delta (l): shard 0 only
  cudaStream_t st = c.stream;
  msm_bases_build<G1>(&c, P.a_set, S.a, S.a_words, P.ma + vk_terms, pre, 0, st);
  msm_bases_build<G1>(&c, P.b1_set, S.b1, S.b1_words, P.ma + vk_terms, pre, 0, st);
  msm_bases_build<G1>(&c, P.l_set, S.l, S.l_words, P.ml + vk_terms / 2, pre, 0, st);
  msm_bases_build<G2>(&c, P.g2, S.b2, S.b2_words, P.ma + vk_terms, pre, 0, st);
  msm_bases_build<G1>(&c, P.h, S.h, S.h_words, P.hn, pre, 0, st);
  B2Z_CUDA(cudaStreamSynchronize(st));
  pk_alloc_scratch(c, P);
  return pk.release();
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

// from / to / den, cyc_rank / cyc_world: the shard of pk_shard (prove_internal.hpp), assembled from the caller's arrays
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
    static_cast<PkShard&>(P) = pk_shard(d->log_domain, m, l, from, to, den, cyc_rank, cyc_world);
    cudaStream_t st = c.stream;
    const bool pre = pk_precompute_fits_slice(P.log_n, m, l, to - from, den);
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
      if (P.cyc_world == 0) {
        out.pts = query + (size_t)limbs * (P.var(skip) - shift);
      } else {
        out.own_pts.resize((size_t)limbs * count);
        for (uint32_t j = 0; j < count;) {               // copy block by block
          const uint64_t q = P.var(skip + j) - shift;
          uint32_t run = 1;
          while (j + run < count && P.var(skip + j + run) - shift == q + run) run++;
          std::memcpy(&out.own_pts[(size_t)limbs * j], query + (size_t)limbs * q, (size_t)limbs * 8 * run);
          j += run;
        }
        out.pts = out.own_pts.data();
      }
      if (inf != nullptr) {
        out.own_inf.assign((count + 7) / 8 + 1, 0);
        for (uint32_t j = 0; j < count; j++) {
          const uint64_t q = P.var(skip + j) - shift;
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
      pack_flags_device(&c, flags.p + P.h_lo, P.hn, words.p, st);
      msm_bases_build<G1>(&c, P.h, dst.p + P.h_lo, words.p, P.hn, pre, 0, st);
      B2Z_CUDA(cudaStreamSynchronize(st));
    }
    pk_alloc_scratch(c, P);
    *out = pk.release();
  });
}

}  // extern "C"

namespace b2z {
namespace {
// copy 0 of a base set (the points as uploaded) and its identity bits, on the host
template <class C>
void download_set(const MsmBases<C>& B, std::vector<typename C::Affine>& pts, std::vector<uint32_t>& words,
                  cudaStream_t st) {
  pts.resize(B.n);
  words.assign((B.n + 31) / 32, 0u);
  if (B.n) B2Z_CUDA(cudaMemcpyAsync(pts.data(), B.points.p, B.n * sizeof(pts[0]), cudaMemcpyDeviceToHost, st));
  if (B.n && B.inf_words.p)
    B2Z_CUDA(cudaMemcpyAsync(words.data(), B.inf_words.p, words.size() * 4, cudaMemcpyDeviceToHost, st));
  B2Z_CUDA(cudaStreamSynchronize(st));
}
inline bool word_bit(const std::vector<uint32_t>& w, uint64_t i) { return (w[i >> 5] >> (i & 31)) & 1; }
// points [from, from + count) of a downloaded set -> caller's limbs + identity bitmap
template <class Affine>
void put_query(const std::vector<Affine>& pts, const std::vector<uint32_t>& words, uint64_t count, uint64_t* out,
               uint8_t* inf) {
  if (count == 0) return;
  std::memcpy(out, pts.data(), count * sizeof(Affine));
  std::memset(inf, 0, (count + 7) / 8);
  for (uint64_t i = 0; i < count; i++)
    if (word_bit(words, i)) inf[i >> 3] |= (uint8_t)(1u << (i & 7));
}
}  // namespace
}  // namespace b2z

extern "C" {

b2z_status b2z_pk_download(b2z_ctx* ctx, const b2z_pk* pk, b2z_pk_arrays* out) {
  return guarded(ctx, [&](Ctx& c) {
    B2Z_REQUIRE(out != nullptr, B2Z_EINVAL, "b2z_pk_download: NULL argument");
    const PkImpl& P = pk_of(c, pk, "b2z_pk_download");
    const uint64_t n = 1ull << P.log_n, m = P.m, l = P.l;
    B2Z_REQUIRE(P.whole(), B2Z_EINVAL,
                "b2z_pk_download: the key is a shard; only whole keys (b2z_pk_upload, b2z_groth16_setup) download");
    B2Z_REQUIRE(out->a_query && out->a_inf && out->b_g1_query && out->b_g1_inf && out->b_g2_query && out->b_g2_inf &&
                    (n == 1 || (out->h_query && out->h_inf)) && (m == l || (out->l_query && out->l_inf)),
                B2Z_EINVAL, "b2z_pk_download: NULL query array");
    cudaStream_t st = c.stream;
    out->num_variables = m;
    out->num_instance = l;
    out->log_domain = P.log_n;
    std::vector<G1::Affine> p1;
    std::vector<G2::Affine> p2;
    std::vector<uint32_t> w;
    download_set<G1>(P.a_set, p1, w, st);                  // [a_query | alpha_1 delta_1]
    put_query(p1, w, m, out->a_query, out->a_inf);
    std::memcpy(out->alpha_g1, &p1[m], sizeof(G1::Affine));
    std::memcpy(out->delta_g1, &p1[m + 1], sizeof(G1::Affine));
    download_set<G1>(P.b1_set, p1, w, st);                 // [b_g1_query | beta_1 delta_1]
    put_query(p1, w, m, out->b_g1_query, out->b_g1_inf);
    std::memcpy(out->beta_g1, &p1[m], sizeof(G1::Affine));
    download_set<G1>(P.l_set, p1, w, st);                  // [l_query | delta_1]
    put_query(p1, w, m - l, out->l_query, out->l_inf);
    download_set<G2>(P.g2, p2, w, st);                     // [b_g2_query | beta_2 delta_2]
    put_query(p2, w, m, out->b_g2_query, out->b_g2_inf);
    std::memcpy(out->beta_g2, &p2[m], sizeof(G2::Affine));
    std::memcpy(out->delta_g2, &p2[m + 1], sizeof(G2::Affine));
    if (n > 1) {                                           // h: bit-reversed, padded to n -> natural order, n - 1 points
      download_set<G1>(P.h, p1, w, st);
      std::vector<G1::Affine> nat(n - 1);
      std::vector<uint32_t> nat_w((n + 31) / 32, 0u);
      for (uint64_t p = 0; p < n; p++) {
        uint64_t j = 0;
        for (uint32_t b = 0; b < P.log_n; b++) j |= ((p >> b) & 1) << (P.log_n - 1 - b);
        if (j >= n - 1) continue;
        nat[j] = p1[p];
        if (word_bit(w, p)) nat_w[j >> 5] |= 1u << (j & 31);
      }
      put_query(nat, nat_w, n - 1, out->h_query, out->h_inf);
    }
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
    stage_host_inputs(c, P, a_evals, b_evals, c_evals, z);
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
    stage_host_inputs(c, P, a_evals, b_evals, c_evals, z);
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
