// A parsed PreparedVerifyingKey (host_pairing.hpp) in the layout of pairing.cuh's per-proof verifier, and the
// call-level checks of Groth16::verify_with_processed_vk.  Shared by b2z_groth16_verify_batch (verify_batch.cu) and
// its host self-check b2z_host_verify_one (hostcheck.cu).
#pragma once
#include <cstring>
#include <vector>

#include "host_pairing.hpp"
#include "pairing.cuh"

namespace b2z {
namespace pairing {

struct FinalParams {
  FrobConsts fc;
  Fq12El alpha_beta;
};

struct KeyArrays {
  std::vector<AffinePoint<Fq>> abc;
  std::vector<uint8_t> abc_inf;
  std::vector<LineCoeffs> lines;           // gamma's kLines, then delta's (zeros for an infinite one)
  bool gamma_inf = true, delta_inf = true;
  FinalParams fp;
};

inline FqEl from_host(const host::Fq& a) {   // same Montgomery radix and little-endian limb order
  FqEl r;
  std::memcpy(r.l, a.l, sizeof(r.l));
  return r;
}
inline Fq2El from_host(const host::Fq2& a) { return Fq2El{from_host(a.c0), from_host(a.c1)}; }

// The errors the single-proof verifier returns for the whole call, whatever the proof: nullptr when there are none.
inline const char* key_error(const host::PreparedVk& k, uint64_t num_inputs) {
  if (num_inputs + 1 != k.gamma_abc_g1.size()) return "num_inputs + 1 differs from the pvk's gamma_abc_g1 count";
  for (const host::G2Prepared* g : {&k.gamma_g2_neg_pc, &k.delta_g2_neg_pc})
    if (!g->inf && g->ell.size() != (size_t)kLines) return "a prepared G2 line list is neither infinite nor 68 long";
  return nullptr;
}

inline KeyArrays key_arrays(const host::PreparedVk& k) {
  KeyArrays a;
  a.abc.resize(k.gamma_abc_g1.size());
  a.abc_inf.resize(k.gamma_abc_g1.size());
  for (size_t j = 0; j < a.abc.size(); j++) {
    a.abc[j] = AffinePoint<Fq>{from_host(k.gamma_abc_g1[j].x), from_host(k.gamma_abc_g1[j].y)};
    a.abc_inf[j] = k.gamma_abc_g1[j].inf ? 1 : 0;
  }
  a.lines.assign(2 * kLines, LineCoeffs{Fq2::zero(), Fq2::zero(), Fq2::zero()});
  const host::G2Prepared* prep[2] = {&k.gamma_g2_neg_pc, &k.delta_g2_neg_pc};
  for (int g = 0; g < 2; g++)
    if (!prep[g]->inf)
      for (int s = 0; s < kLines; s++) {
        const host::EllCoeff& e = prep[g]->ell[s];
        a.lines[g * kLines + s] = LineCoeffs{from_host(e.c0), from_host(e.c1), from_host(e.c2)};
      }
  a.gamma_inf = k.gamma_g2_neg_pc.inf;
  a.delta_inf = k.delta_g2_neg_pc.inf;
  a.fp.fc = frobenius_consts();
  const host::Fq2* ab = &k.alpha_g1_beta_g2.c0.c0;
  Fq2El* dst = &a.fp.alpha_beta.c0.c0;
  for (int i = 0; i < 6; i++) dst[i] = from_host(ab[i]);
  return a;
}

// The view the per-proof code reads, over arrays at abc / abc_inf / lines (device or host copies of a KeyArrays).
inline KeyView key_view(const KeyArrays& a, const AffinePoint<Fq>* abc, const uint8_t* abc_inf,
                        const LineCoeffs* lines) {
  KeyView v;
  v.abc = abc;
  v.abc_inf = abc_inf;
  v.gamma_lines = lines;
  v.delta_lines = lines + kLines;
  v.num_inputs = (uint32_t)(a.abc.size() - 1);
  v.gamma_inf = a.gamma_inf ? 1u : 0u;
  v.delta_inf = a.delta_inf ? 1u : 0u;
  return v;
}

}  // namespace pairing
}  // namespace b2z
