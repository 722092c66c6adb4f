// b2z_groth16_verify_batch: Groth16::verify_with_processed_vk for many proofs against one prepared verifying key,
// one verdict per proof (row f4 on the GPU).  The pvk is parsed on the host by host_pairing.hpp's pvk_deserialize
// and uploaded once per call; proofs and inputs go through the device in fixed-size chunks, one proof per thread,
// in three kernels so that each keeps its own register budget:
//   verify_decode_kernel     decompress + validate A, B, C; inputs to canonical form; the prepared-inputs sum
//   verify_miller_kernel     the three-pair Miller loop (B's lines on the fly, gamma's and delta's from the key)
//   verify_final_exp_kernel  final exponentiation, comparison with alpha_g1_beta_g2 -> 1 / 0 / -1
// The per-thread code is pairing.cuh's, which hostcheck.cu also runs on the host (b2z_host_verify_one).
#include "api_glue.hpp"
#include "msm.hpp"
#include "verify_key.hpp"

namespace b2z {
namespace {

using pairing::Fq12El;
using pairing::FinalParams;
using pairing::KeyView;
using pairing::LineCoeffs;
using pairing::ProofPoints;

constexpr uint32_t kThreads = 128;
constexpr uint64_t kChunk = 1u << 16;      // proofs per pass through the device: bounds device memory for any count

__global__ void __launch_bounds__(kThreads) verify_decode_kernel(const uint8_t* __restrict__ proofs,
                                                                 const FrEl* __restrict__ inputs, KeyView k,
                                                                 uint32_t n, ProofPoints* __restrict__ pts) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  pairing::verify_decode(proofs + 192ull * i, inputs + (uint64_t)k.num_inputs * i, k, &pts[i]);
}

__global__ void __launch_bounds__(kThreads) verify_miller_kernel(const ProofPoints* __restrict__ pts, KeyView k,
                                                                 uint32_t n, Fq12El* __restrict__ f) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const ProofPoints p = pts[i];
  if (p.flags & pairing::PT_MALFORMED) return;
  pairing::verify_miller(p, k, &f[i]);
}

__global__ void __launch_bounds__(kThreads) verify_final_exp_kernel(const ProofPoints* __restrict__ pts,
                                                                    const Fq12El* __restrict__ f, FinalParams fp,
                                                                    uint32_t n, int32_t* __restrict__ results) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  if (pts[i].flags & pairing::PT_MALFORMED) { results[i] = -1; return; }
  results[i] = pairing::verify_final(f[i], fp.alpha_beta, fp.fc);
}

void verify_batch(Ctx& c, const uint8_t* pvk, uint64_t pvk_len, const uint64_t* public_inputs, uint64_t num_inputs,
                  const uint8_t* proofs, uint64_t count, int32_t* results) {
  B2Z_REQUIRE(num_inputs <= pairing::kMaxInputs, B2Z_ESIZE, "b2z_groth16_verify_batch: more than 1024 public inputs");
  host::PreparedVk k;
  B2Z_REQUIRE(host::pvk_deserialize(pvk, pvk_len, &k), B2Z_EINVAL, "b2z_groth16_verify_batch: malformed pvk");
  const char* bad = pairing::key_error(k, num_inputs);
  B2Z_REQUIRE(bad == nullptr, B2Z_EINVAL, std::string("b2z_groth16_verify_batch: ") + (bad ? bad : ""));

  // the key, once per call
  const pairing::KeyArrays ka = pairing::key_arrays(k);
  const cudaStream_t st = c.stream;
  DevBuf<AffinePoint<Fq>> d_abc(ka.abc.size());
  DevBuf<uint8_t> d_abc_inf(ka.abc_inf.size());
  DevBuf<LineCoeffs> d_lines(ka.lines.size());
  B2Z_CUDA(cudaMemcpyAsync(d_abc.p, ka.abc.data(), ka.abc.size() * sizeof(ka.abc[0]), cudaMemcpyHostToDevice, st));
  B2Z_CUDA(cudaMemcpyAsync(d_abc_inf.p, ka.abc_inf.data(), ka.abc_inf.size(), cudaMemcpyHostToDevice, st));
  B2Z_CUDA(cudaMemcpyAsync(d_lines.p, ka.lines.data(), ka.lines.size() * sizeof(ka.lines[0]), cudaMemcpyHostToDevice,
                           st));
  const KeyView kv = pairing::key_view(ka, d_abc.p, d_abc_inf.p, d_lines.p);

  const uint64_t chunk = count < kChunk ? count : kChunk;
  DevBuf<uint8_t> d_proofs(chunk * 192);
  DevBuf<FrEl> d_inputs(chunk * num_inputs);
  DevBuf<ProofPoints> d_pts(chunk);
  DevBuf<Fq12El> d_f(chunk);
  DevBuf<int32_t> d_res(chunk);
  for (uint64_t at = 0; at < count; at += chunk) {
    const uint32_t n = (uint32_t)(count - at < chunk ? count - at : chunk);
    B2Z_CUDA(cudaMemcpyAsync(d_proofs.p, proofs + 192 * at, 192ull * n, cudaMemcpyHostToDevice, st));
    if (num_inputs)
      B2Z_CUDA(cudaMemcpyAsync(d_inputs.p, public_inputs + 4 * num_inputs * at, 32ull * num_inputs * n,
                               cudaMemcpyHostToDevice, st));
    verify_decode_kernel<<<nblocks(n, kThreads), kThreads, 0, st>>>(d_proofs.p, d_inputs.p, kv, n, d_pts.p);
    B2Z_LAUNCHED(&c);
    verify_miller_kernel<<<nblocks(n, kThreads), kThreads, 0, st>>>(d_pts.p, kv, n, d_f.p);
    B2Z_LAUNCHED(&c);
    verify_final_exp_kernel<<<nblocks(n, kThreads), kThreads, 0, st>>>(d_pts.p, d_f.p, ka.fp, n, d_res.p);
    B2Z_LAUNCHED(&c);
    B2Z_CUDA(cudaMemcpyAsync(results + at, d_res.p, 4ull * n, cudaMemcpyDeviceToHost, st));
  }
  B2Z_CUDA(cudaStreamSynchronize(st));
}

}  // namespace
}  // namespace b2z

extern "C" b2z_status b2z_groth16_verify_batch(b2z_ctx* ctx, const uint8_t* pvk, uint64_t pvk_len,
                                               const uint64_t* public_inputs, uint64_t num_inputs,
                                               const uint8_t* proofs, uint64_t count, int32_t* results) {
  if (ctx == nullptr) return B2Z_EINVAL;
  if (count == 0) return B2Z_OK;
  if (pvk == nullptr || proofs == nullptr || results == nullptr || (num_inputs && public_inputs == nullptr))
    return B2Z_EINVAL;
  return b2z::guarded(ctx, [&](b2z::Ctx& c) {
    b2z::verify_batch(c, pvk, pvk_len, public_inputs, num_inputs, proofs, count, results);
  });
}
