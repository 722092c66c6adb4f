// Host-side self checks: the device limb algorithms (mont.cuh, ec.cuh, the MSM
// digit recoding) run here through the carry-flag emulation of ptx.cuh, so the
// CPU-only test suite can compare them with the oracle.  None of this is used
// by the proving path.
#include <cstring>

#include <vector>

#include "accum_affine.cuh"
#include "host_fq.hpp"
#include "inv_gcd.cuh"
#include "msm.hpp"

using namespace b2z;

namespace {

template <class F>
int field_op(int op, const uint32_t* a, const uint32_t* b, uint32_t* out) {
  typename F::El x, y, r;
  std::memcpy(x.l, a, sizeof(x.l));
  if (b) std::memcpy(y.l, b, sizeof(y.l));
  switch (op) {
    case 0: r = F::mul_safe(x, y); break;
    case 1: r = F::add(x, y); break;
    case 2: r = F::sub(x, y); break;
    case 3: r = F::reduce(x); break;
    case 4: r = F::reduce(F::inv(x)); break;
    case 5: r = F::mul(x, y); break;   // raw product: caller honours the operand precondition
    default: return -1;
  }
  std::memcpy(out, r.l, sizeof(r.l));
  return 0;
}

template <class C>
int point_sum(const uint32_t* points, const uint8_t* neg, uint32_t n, uint32_t* out_affine) {
  using Affine = typename C::Affine;
  typename C::Xyzz acc = C::identity();
  typename C::Xyzz acc2 = C::identity();
  for (uint32_t i = 0; i < n; i++) {
    Affine p;
    std::memcpy(&p, points + (size_t)i * (sizeof(Affine) / 4), sizeof(Affine));
    if (neg && neg[i]) p = C::neg(p);
    acc = C::madd(acc, p);                       // mixed addition path
    acc2 = C::add(acc2, C::from_affine(p));      // general addition path
  }
  bool inf = false, inf2 = false;
  const Affine r = C::to_affine(acc, &inf);
  const Affine r2 = C::to_affine(acc2, &inf2);
  if (inf != inf2 || std::memcmp(&r, &r2, sizeof(Affine)) != 0) return -1;   // the two paths must agree
  std::memcpy(out_affine, &r, sizeof(Affine));
  return inf ? 1 : 0;
}

// The batched-affine accumulation of accum_affine.cuh, one emulated thread per segment, checked bucket by bucket
// against the XYZZ running sum: bucket_out[b] + (partial entries keyed b) must equal the naive sum of the bucket's
// references.  Returns the number of buckets that differ (or -2 when the partial list is not sorted by key).
template <class C>
int accum_affine_check(const uint32_t* points_raw, const uint32_t* sorted, const uint32_t* offsets, uint32_t nbuckets,
                       uint32_t nseg, uint32_t cap_override, uint32_t* rounds_hint) {
  using Affine = typename C::Affine;
  using Xyzz = typename C::Xyzz;
  using El = typename C::El;
  const Affine* points = reinterpret_cast<const Affine*>(points_raw);
  std::vector<Xyzz> bucket_out(nbuckets, C::identity()), part_pts(2 * (size_t)nseg, C::identity());
  std::vector<uint32_t> part_keys(2 * (size_t)nseg, aff::kEmptyKey);
  uint32_t maxrun = 0;
  (void)cap_override;
  std::vector<Affine> b0, b1;
  std::vector<uint32_t> k0, k1;
  std::vector<El> pref;
  std::vector<uint4> desc;
  for (uint32_t seg = 0; seg < nseg; seg++) {
    aff::Segment<C> G(offsets, nbuckets, nseg, seg, bucket_out.data(), part_keys.data(), part_pts.data(), &maxrun);
    if (!G.active) {
      G.close_empty();
      continue;
    }
    const uint32_t cap = G.seg_len;
    b0.resize(cap + 1); b1.resize(cap + 1);
    k0.resize(cap + 1); k1.resize(cap + 1);
    pref.resize(cap / 2 + 2); desc.resize(cap / 2 + 2);
    aff::Scratch<C> S;
    S.pts[0] = b0.data(); S.pts[1] = b1.data();
    S.keys[0] = k0.data(); S.keys[1] = k1.data();
    S.pref = pref.data(); S.desc = desc.data();
    aff::accum_segment<C>(points, sorted, offsets, G, S);
  }
  if (rounds_hint) {                       // [0] maxrun, [1..6] the emulation's counters (accum_affine.cuh)
    rounds_hint[0] = maxrun;
    for (int i = 0; i < 6; i++) { rounds_hint[1 + i] = (uint32_t)aff::host_stats()[i]; aff::host_stats()[i] = 0; }
  }
  uint32_t prev = 0;
  for (uint32_t k : part_keys) {
    if (k == 0xffffffffu) continue;
    if (k < prev || k >= nbuckets) return -2;
    prev = k;
  }
  int bad = 0;
  for (uint32_t b = 0; b < nbuckets; b++) {
    Xyzz want = C::identity();
    for (uint32_t i = offsets[b]; i < offsets[b + 1]; i++) {
      Affine p = points[sorted[i] & 0x7fffffffu];
      if (sorted[i] & 0x80000000u) p = C::neg(p);
      want = C::madd(want, p);
    }
    Xyzz got = bucket_out[b];
    for (size_t i = 0; i < part_keys.size(); i++)
      if (part_keys[i] == b) got = C::add(got, part_pts[i]);
    bool i1 = false, i2 = false;
    const Affine w = C::to_affine(want, &i1), g = C::to_affine(got, &i2);
    if (i1 != i2 || std::memcmp(&w, &g, sizeof(Affine)) != 0) bad++;
  }
  return bad;
}

}  // namespace

extern "C" {

int b2z_host_accum_affine(int group, const uint32_t* points, const uint32_t* sorted, const uint32_t* offsets,
                          uint32_t nbuckets, uint32_t nseg, uint32_t cap, uint32_t* maxrun_out) {
  if (points == nullptr || sorted == nullptr || offsets == nullptr || nseg == 0) return -1;
  return group == 1 ? accum_affine_check<G1>(points, sorted, offsets, nbuckets, nseg, cap, maxrun_out)
                    : accum_affine_check<G2>(points, sorted, offsets, nbuckets, nseg, cap, maxrun_out);
}

int b2z_host_field_op(int field, int op, const uint32_t* a, const uint32_t* b, uint32_t* out) {
  if (a == nullptr || out == nullptr) return -1;
  return field == 0 ? field_op<Fr>(op, a, b, out) : field_op<Fq>(op, a, b, out);
}

int b2z_host_point_sum(int group, const uint32_t* points, const uint8_t* neg, uint32_t n, uint32_t* out_affine) {
  if (out_affine == nullptr || (n && points == nullptr)) return -1;
  return group == 1 ? point_sum<G1>(points, neg, n, out_affine) : point_sum<G2>(points, neg, n, out_affine);
}

// division-step inversion of an Fq element in Montgomery form (inv_gcd.cuh); returns the number of 30-step batches
int b2z_host_fq_inv_gcd(const uint32_t* a, uint32_t* out) {
  if (a == nullptr || out == nullptr) return -1;
  FqEl x;
  std::memcpy(x.l, a, sizeof(x.l));
  int batches = 0;
  const FqEl r = Fq::reduce(gcdinv::inv(x, &batches));
  std::memcpy(out, r.l, sizeof(r.l));
  return batches;
}

uint32_t b2z_host_msm_digits(const uint32_t scalar[8], uint32_t c, int32_t* digits) {
  DigitCfg cfg;
  cfg.c = c;
  cfg.windows = msm_windows(c);
  cfg.nb = 1u << (c - 1);
  cfg.n = 1;
  cfg.precomputed = 0;
  FrEl k;
  std::memcpy(k.l, scalar, 32);
  for (uint32_t w = 0; w < cfg.windows; w++) digits[w] = 0;
  for_each_digit(k, cfg, [&](uint32_t w, uint32_t v, bool neg) { digits[w] = neg ? -(int32_t)v : (int32_t)v; });
  return cfg.windows;
}

int b2z_host_planes_horner(int group, const uint32_t* planes_xyzz, uint32_t nplanes, uint32_t chunk_log, uint8_t* out) {
  if (out == nullptr || (nplanes && planes_xyzz == nullptr)) return -1;
  if (group == 1) host::g1_serialize(out, host::g1_planes_horner(planes_xyzz, nplanes, chunk_log));
  else host::g2_serialize(out, host::g2_planes_horner(planes_xyzz, nplanes, chunk_log));
  return 0;
}

uint32_t b2z_host_msm_window_bits(uint64_t n, int precomputed) { return msm_pick_c(n, precomputed != 0); }

}  // extern "C"
