// Bucket (Pippenger) multi-scalar multiplication -- internal interface.
#pragma once
#include "common.hpp"
#include "ec.cuh"

namespace b2z {

// Device-resident base set prepared for repeated MSMs.
//   generic     : `points` holds n affine points; every signed window keeps its
//                 own 2^(c-1) buckets and the window sums are combined by
//                 c doublings each (Horner).
//   precomputed : `points` holds `windows` copies, copy w = 2^(c*w) * P_i, so
//                 ALL windows share one bucket set and no doublings remain.
//                 This trades HBM capacity (windows x the key size; a 2^22
//                 Groth16 key is ~23 GB of the 180 GB) for the Horner tail and
//                 for windows-1 of the bucket reductions.
template <class C>
struct MsmBases {
  DevBuf<typename C::Affine> points;
  DevBuf<uint32_t> inf_words;     // bit i set => base i is the identity (may be empty)
  uint32_t n = 0;                 // number of bases (per copy)
  uint32_t c = 0;                 // window bits
  uint32_t windows = 0;
  bool precomputed = false;
};

struct DigitCfg {
  uint32_t c;
  uint32_t windows;
  uint32_t nb;           // 2^(c-1) buckets per window
  uint32_t n;            // number of bases
  uint32_t precomputed;  // shared buckets, point index = w*n + i
};

// Signed digits d_w in [-2^(c-1), 2^(c-1)) for w < windows-1, the top window
// keeps its carry (non-negative, <= 2^(c-1)); msm_windows() guarantees it fits.
template <class Emit>
B2Z_HD void for_each_digit(const FrEl& k, const DigitCfg& cfg, Emit&& emit) {
  uint32_t carry = 0;
  const uint32_t mask = (1u << cfg.c) - 1;
  for (uint32_t w = 0; w < cfg.windows; w++) {
    const uint32_t bit = w * cfg.c;
    const uint32_t limb = bit >> 5, sh = bit & 31;
    uint32_t raw = 0;
    if (limb < 8) {
      uint64_t two = k.l[limb];
      if (limb + 1 < 8) two |= (uint64_t)k.l[limb + 1] << 32;
      raw = (uint32_t)(two >> sh) & mask;
    }
    uint32_t v = raw + carry;
    carry = 0;
    bool neg = false;
    if (w + 1 < cfg.windows && v > cfg.nb) {   // v in (2^(c-1), 2^c]  ->  v - 2^c, carry
      v = (1u << cfg.c) - v;
      neg = true;
      carry = 1;
    }
    if (v != 0) emit(w, v, neg);
  }
}

// Scratch arenas: one per concurrently running MSM (indexed by `slot`).
struct MsmArena {
  DevBuf<uint32_t> hist, offsets, cursor, tile_sums, sorted;
  DevBuf<uint32_t> keys[2], state;
  DevBuf<uint8_t> buckets, parts[2], chunks[3], wsums;
  // batched-affine accumulation (accum_affine.cuh): entry lists, their keys, prefix products, descriptors
  DevBuf<uint8_t> aff_pts, aff_pref;
  DevBuf<uint32_t> aff_keys;
  DevBuf<uint4> aff_desc;
};
struct MsmScratch {
  MsmArena slot[8];
};

// Fixed-base tables: [window][digit], 8-bit windows.  The context caches the standard generators' tables; key
// generation with a caller's generator builds its own (32 x 256 points).
constexpr uint32_t kFbWindows = 32, kFbEntries = 256;
template <class C>
struct FbTable {
  DevBuf<typename C::Affine> table;
};
struct FixedBaseTables {
  FbTable<G1> g1;
  FbTable<G2> g2;
  template <class C> FbTable<C>& get();
};
template <> inline FbTable<G1>& FixedBaseTables::get<G1>() { return g1; }
template <> inline FbTable<G2>& FixedBaseTables::get<G2>() { return g2; }

// Window size / count rules.
uint32_t msm_pick_c(uint64_t n, bool precomputed);
uint32_t msm_windows(uint32_t c);

// Builds a base set from n affine points already on the device (copied).
template <class C>
void msm_bases_build(Ctx* ctx, MsmBases<C>& out, const typename C::Affine* d_points, const uint32_t* d_inf_words,
                     uint32_t n, bool precompute, uint32_t c_override, cudaStream_t st);

// result (device, one XYZZ point) = sum_i scalars[i] * P_i.
// scalars: canonical 8 x u32 little-endian; index i < n_main reads main[i], the
// rest reads tail[i - n_main] (lets the prover append its {1, r} / {1, s} terms
// without copying z).  `slot` selects a scratch arena so MSMs on different
// streams can overlap.
template <class C>
void msm_run(Ctx* ctx, int slot, const MsmBases<C>& bases, const FrEl* d_scalars_main, uint32_t n_main,
             const FrEl* d_scalars_tail, typename C::Xyzz* d_result, cudaStream_t st);

// The same in two halves, so that a proof can run all the light work (sorts) first and then chain
// the GPU-filling accumulations: msm_sort = digits + counting sort; msm_finish = accumulate (after
// `wait_before_accum`, signalling `record_after_accum` when the accumulation kernel is done) + reduce.
template <class C>
void msm_sort(Ctx* ctx, int slot, const MsmBases<C>& bases, const FrEl* d_scalars_main, uint32_t n_main,
              const FrEl* d_scalars_tail, cudaStream_t st);
//
// `host_planes` (optional, pinned): the last, strictly serial step of the bucket reduction -- a Horner
// pass of ~2 point operations per bit plane -- is then left to the CALLER's CPU, which does a point
// operation in 0.5 us where a lone GPU warp needs 6 us: the bit-plane sums (nplanes XYZZ points, 2.5 KB
// for G1) are copied to `host_planes->host` on `st` instead of reducing them into d_result, and the
// caller finishes with host::planes_horner (host_fq.hpp) after synchronising.
constexpr uint32_t kMsmMaxPlanes = 32;
constexpr uint32_t kMsmChunkLog = 3;     // buckets per running-sum chunk = 8
struct MsmHostPlanes {
  void* host = nullptr;       // pinned, kMsmMaxPlanes * sizeof(Xyzz)
  uint32_t nplanes = 0;       // set by msm_finish (0 = the sum is the identity)
};
template <class C>
void msm_finish(Ctx* ctx, int slot, const MsmBases<C>& bases, typename C::Xyzz* d_result, cudaStream_t st,
                cudaEvent_t wait_before_accum, cudaEvent_t record_after_accum, MsmHostPlanes* host_planes = nullptr);

void msm_release_scratch(Ctx* ctx);

// r (device XYZZ[count]) -> affine limbs + infinity flags on the host side layout
template <class C>
void xyzz_to_affine_device(Ctx* ctx, const typename C::Xyzz* d_in, typename C::Affine* d_out, uint32_t* d_inf, uint32_t count,
                           cudaStream_t st);

// Fr Montgomery -> canonical integers (scalars for the MSM), out-of-place.
void fr_from_mont_device(Ctx* ctx, const FrEl* in, FrEl* out, size_t n, cudaStream_t st);

// identity flags (one u32 per point, non-zero = identity) -> bitmap words (bit i of word i / 32), n points
void pack_flags_device(Ctx* ctx, const uint32_t* d_flags, uint32_t n, uint32_t* d_words, cudaStream_t st);

// blocks of `threads` that cover n items
inline uint32_t nblocks(uint64_t n, uint32_t threads) { return (uint32_t)((n + threads - 1) / threads); }

// table for the generator `gen` (affine, Montgomery limbs, not the identity)
template <class C>
void fb_build(Ctx* ctx, FbTable<C>& t, const typename C::Affine& gen, cudaStream_t st);
// the standard generator's table, built on first use and cached in the context
template <class C>
const FbTable<C>& fb_standard_table(Ctx* ctx, cudaStream_t st);
// out[i] = scalars[i] * G for the table's G: affine points, identity bitmap words; scalars canonical.  Returns when done.
template <class C>
void fixed_base_mul(Ctx* ctx, const FbTable<C>& t, const FrEl* d_scalars, typename C::Affine* d_out,
                    uint32_t* d_inf_words, uint32_t n, cudaStream_t st);

// out[i] = scalars[i] * G (standard generator), affine; scalars canonical.
void g1_fixed_base_mul_device(Ctx* ctx, const FrEl* d_scalars, G1::Affine* d_out, uint32_t* d_inf_words, uint32_t n,
                              cudaStream_t st);
void g2_fixed_base_mul_device(Ctx* ctx, const FrEl* d_scalars, G2::Affine* d_out, uint32_t* d_inf_words, uint32_t n,
                              cudaStream_t st);

}  // namespace b2z
