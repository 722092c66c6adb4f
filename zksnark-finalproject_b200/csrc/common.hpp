// Library-internal declarations shared by the translation units of libb200zk.
#pragma once
#include <cuda_runtime.h>

#include <cstdint>
#include <cstdio>
#include <map>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/b200zk.h"
#include "mont.cuh"

namespace b2z {

struct StatusError {
  b2z_status code;
  std::string msg;
};

#define B2Z_CUDA(expr)                                                                     \
  do {                                                                                     \
    cudaError_t e__ = (expr);                                                              \
    if (e__ != cudaSuccess)                                                                \
      throw ::b2z::StatusError{e__ == cudaErrorMemoryAllocation ? B2Z_ENOMEM : B2Z_ECUDA,  \
                               std::string(#expr) + ": " + cudaGetErrorString(e__)};       \
  } while (0)

// after every kernel launch: count it and surface launch errors
#define B2Z_LAUNCHED(ctx_ptr)              \
  do {                                     \
    (ctx_ptr)->launches++;                 \
    B2Z_CUDA(cudaGetLastError());          \
  } while (0)

#define B2Z_REQUIRE(cond, code, text)                                  \
  do {                                                                 \
    if (!(cond)) throw ::b2z::StatusError{code, std::string(text)};    \
  } while (0)

// RAII device buffer.
template <class T>
struct DevBuf {
  T* p = nullptr;
  size_t n = 0;
  DevBuf() = default;
  explicit DevBuf(size_t count) { alloc(count); }
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  DevBuf(DevBuf&& o) noexcept : p(o.p), n(o.n) { o.p = nullptr; o.n = 0; }
  DevBuf& operator=(DevBuf&& o) noexcept {
    if (this != &o) { release(); p = o.p; n = o.n; o.p = nullptr; o.n = 0; }
    return *this;
  }
  ~DevBuf() { release(); }
  void alloc(size_t count) {
    release();
    n = count;
    if (count) B2Z_CUDA(cudaMalloc(&p, count * sizeof(T)));
  }
  void ensure(size_t count) { if (count > n) alloc(count); }
  void release() { if (p) cudaFree(p); p = nullptr; n = 0; }
};

// ---------------------------------------------------------------------------
// NTT (ntt.cu)
// ---------------------------------------------------------------------------
enum TwKind { TW_FWD = 0, TW_INV = 1, TW_COSET_FWD = 2, TW_COSET_INV = 3, TW_KINDS = 4 };

// Per-domain-size twiddle tables, level-major: level L (butterfly half-size 2^L)
// occupies entries [2^L - 1, 2^(L+1) - 1); n - 1 entries per kind.
struct NttDomain {
  uint32_t log_n = 0;
  DevBuf<FrEl> tw[TW_KINDS];
  FrEl n_inv;            // n^-1                     (Montgomery)
  FrEl wm_k1, wm_k2;     // n^-3 Z^-1, n^-2 Z^-1     (witness-map pointwise constants)
};

// ---------------------------------------------------------------------------
// Profiling spans (CUDA events on the launching stream) and launch counting
// ---------------------------------------------------------------------------
enum Phase {
  PH_NTT_PASS = 0,      // every NTT pass kernel            units: field elements
  PH_WM_POINTWISE = 1,  // witness-map pointwise kernel     units: field elements
  PH_MSM_SORT = 2,      // digits + counting sort           units: scalars
  PH_MSM_ACCUM_G1 = 3,  // bucket accumulation kernel, G1   units: mixed additions
  PH_MSM_ACCUM_G2 = 4,  // bucket accumulation kernel, G2   units: mixed additions
  PH_MSM_REDUCE = 5,    // partial lists, bucket reduction, window combine
  PH_R1CS_EVAL = 6,     // constraint-row evaluation (CSR SpMV)
  PH_MSM_ACCUM_AFFINE = 7,  // the accumulation launches (G1 or G2, also counted above) that took the batched-affine kernel
  PH_COUNT = 8
};

constexpr uint32_t kUnitsPool = 4096;
struct ProfileSpan {
  int phase;
  cudaEvent_t start, stop;
  uint64_t units;
  uint32_t* units_pinned;   // optional: filled by an async D2H copy (actual entry count)
};

struct Ctx;
struct ProfileScope {
  Ctx* ctx;
  cudaStream_t st;
  int idx = -1;
  ProfileScope(Ctx* c, int phase, cudaStream_t s, uint64_t units, const uint32_t* d_units = nullptr);
  ~ProfileScope();
};

const NttDomain& ntt_domain(Ctx* ctx, uint32_t log_n);
const FrEl* ntt_twiddles(Ctx* ctx, uint32_t log_n, TwKind kind, cudaStream_t st);

// natural -> bit-reversed
void ntt_dif(Ctx* ctx, const FrEl* tw, FrEl* data, uint32_t log_n, cudaStream_t st);
// bit-reversed -> natural
void ntt_dit(Ctx* ctx, const FrEl* tw, FrEl* data, uint32_t log_n, cudaStream_t st);
// DIF with tw_a then DIT with tw_b (natural -> natural), low stages fused in one kernel
void ntt_dif_dit(Ctx* ctx, const FrEl* tw_a, const FrEl* tw_b, FrEl* data, uint32_t log_n, cudaStream_t st);
// in-place bit-reversal permutation; if scale != nullptr every element is also
// multiplied by *scale (host value); if pw_lo/pw_hi != nullptr additionally by
// pw_lo[i & 1023] * pw_hi[i >> 10] with i the NATURAL (destination) index.
void ntt_bitrev(Ctx* ctx, FrEl* data, uint32_t log_n, const FrEl* scale, const FrEl* pw_lo, const FrEl* pw_hi, cudaStream_t st);
// data[i] *= pw_lo[i & 1023] * pw_hi[i >> 10]
void ntt_scale_powers(Ctx* ctx, FrEl* data, uint32_t log_n, const FrEl* pw_lo, const FrEl* pw_hi, cudaStream_t st);
// out[j] = base^j, j < count
void fr_pow_table(Ctx* ctx, FrEl* out, const FrEl& base, uint32_t count, cudaStream_t st);
// a <- a*b*k1 - c*k2   (witness-map pointwise step, constants folded)
void wm_pointwise(Ctx* ctx, FrEl* a, const FrEl* b, const FrEl* c, uint32_t log_n, const FrEl& k1, const FrEl& k2, cudaStream_t st);
// canonicalise (lazy -> [0, p)) in place
void fr_canonicalize(Ctx* ctx, FrEl* data, size_t n, cudaStream_t st);

// 32-bit multiply-add issue rates (ops/s): plain IMAD and the carry-chained wide form
void measure_int_peak(Ctx* ctx, double* imad_per_s, double* imad_wide_per_s);

// Full witness map on device buffers a, b, c (natural order, destroyed); h is
// left in `a`, in bit-reversed order if !natural_out.
void witness_map_device(Ctx* ctx, FrEl* a, FrEl* b, FrEl* c, uint32_t log_n, bool natural_out, cudaStream_t st);
// its two halves (the first one per input vector), for the distributed witness map of the sharded prover
void witness_map_transform(Ctx* ctx, FrEl* x, uint32_t log_n, cudaStream_t st);
void witness_map_transform3(Ctx* ctx, FrEl* a, FrEl* b, FrEl* c, uint32_t log_n, cudaStream_t st);

// Tile-sharded witness map over W = 2^wbits ranks (ntt.cu).  x / y: this rank's local vectors (a, b, c) in the
// column-owned / row-owned layout, n / W elements each; peer_x / peer_y [vector][rank]: the same buffers of
// every rank (peer-mapped device pointers; [..][me] = own).
struct NttDist {
  uint32_t wbits = 0, me = 0;
  FrEl* x[3] = {nullptr, nullptr, nullptr};
  FrEl* y[3] = {nullptr, nullptr, nullptr};
  FrEl* peer_x[3][8] = {};
  FrEl* peer_y[3][8] = {};
};
bool ntt_dist_supported(uint32_t log_n, uint32_t wbits);
uint32_t ntt_dist_col_bits(uint32_t log_n, uint32_t wbits);   // position of the ownership bits of the column-owned layout
void wm_dist_step1(Ctx* ctx, const NttDist& D, uint32_t log_n, cudaStream_t st);   // writes peers' y
void wm_dist_step2(Ctx* ctx, const NttDist& D, uint32_t log_n, cudaStream_t st);   // reads y, writes peers' x
void wm_dist_step3(Ctx* ctx, const NttDist& D, uint32_t log_n, cudaStream_t st);   // reads x, writes peers' y[0]
void wm_dist_step4(Ctx* ctx, const NttDist& D, uint32_t log_n, cudaStream_t st);   // reads y[0]: h chunk, canonical
void witness_map_quotient(Ctx* ctx, FrEl* a, const FrEl* b, const FrEl* c, uint32_t log_n, bool natural_out, cudaStream_t st);

// ---------------------------------------------------------------------------
// Context
// ---------------------------------------------------------------------------
struct Ctx {
  int device = 0;
  std::mutex mu;                       // one in-flight call per context (see include/b200zk.h)
  cudaStream_t stream = nullptr;
  cudaStream_t aux[4] = {nullptr, nullptr, nullptr, nullptr};
  std::map<uint32_t, NttDomain> domains;
  bool ntt_attr_set[6] = {false, false, false, false, false, false};
  bool msm_attr_set[2] = {false, false};   // the G2 accumulation kernels' shared-memory limit: XYZZ, batched-affine
  bool profile = false;
  std::vector<ProfileSpan> spans;
  // pools, so that an enabled profiler costs the launching thread two event records per span and nothing else
  // (creating events and page-locked words inside the timed region delayed the launches by milliseconds)
  std::vector<cudaEvent_t> event_pool;
  uint32_t* units_pool = nullptr;      // page-locked, kUnitsPool words
  uint32_t units_used = 0;
  std::mutex span_mu;                  // spans are appended from the single calling thread; guards reads
  uint64_t launches = 0;               // kernels launched through this context
  void* msm_scratch = nullptr;         // MsmScratch arenas (msm.cu)
  void* fixed_base = nullptr;          // generator tables (msm.cu)
  std::string last_error;
};

}  // namespace b2z
