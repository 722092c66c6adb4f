// Groth16 key generation on the device -- ark_groth16::generator::generate_parameters_with_qap::<LibsnarkReduction>
// (reached from Groth16::setup, reference call sites matrix_proof.rs:128-131, fibbonaci_handler.rs:107,
// prime_snark.rs:111-115) for matrices uploaded with b2z_r1cs_upload, the toxic waste and the generators the caller's:
//
//   L_i    = Z(tau)/n w^i / (tau - w^i)                       i < nc + l   (Lagrange coefficients at tau)
//   A_j    = sum_i A[i][j] L_i  (+ L_{nc+j} for j < l)         B_j, C_j likewise, without the instance term
//   a_query = A_j g1    b_g1_query = B_j g1    b_g2_query = B_j g2
//   l_query = (beta A_j + alpha B_j + C_j)/delta g1   j >= l     gamma_abc = (...)/gamma g1   j < l
//   h_query = tau^i Z(tau)/delta g1   i < n - 1
//
// Everything stays in device memory: the scalars go to the fixed-base multiplication as canonical integers, the h
// scalars straight to their bit-reversed position of the prover's n-padded H set, and the point sets to the key
// assembly that b2z_pk_upload uses (prove.cu: pk_from_device_sets).  Only the verifying key comes back to the host.
#include <cstring>

#include "api_glue.hpp"
#include "host_fr.hpp"
#include "host_pairing.hpp"
#include "msm.hpp"
#include "prove_internal.hpp"

namespace b2z {
namespace {

template <class T> __device__ __forceinline__ T ld_vec(const T* p) { return *p; }   // FrEl: 16-byte aligned
template <class T> __device__ __forceinline__ void st_vec(T* p, const T& v) { *p = v; }
// canonical in, canonical out
__device__ __forceinline__ FrEl fmul(const FrEl& a, const FrEl& b) { return Fr::reduce(Fr::mul(a, b)); }
__device__ __forceinline__ FrEl fadd(const FrEl& a, const FrEl& b) { return Fr::reduce(Fr::add(a, b)); }
__device__ __forceinline__ FrEl fsub(const FrEl& a, const FrEl& b) { return Fr::reduce(Fr::sub(a, b)); }
// x^i from the tables lo[k] = x^k (k < 1024), hi[k] = x^(1024 k)
__device__ __forceinline__ FrEl pow_from_tables(const FrEl* lo, const FrEl* hi, uint32_t i) {
  return fmul(ld_vec(lo + (i & 1023)), ld_vec(hi + (i >> 10)));
}

// ---- 1. Lagrange coefficients at tau: each thread batch-inverts the (tau - w^i) of its chunk with one inversion;
// the prefix products wait in `out`
constexpr uint32_t kLagChunk = 64;
__global__ void __launch_bounds__(128)
    setup_lagrange_kernel(const FrEl* __restrict__ wlo, const FrEl* __restrict__ whi, const FrEl tau, const FrEl zn,
                          uint32_t count, FrEl* out) {
  const uint32_t i0 = (blockIdx.x * blockDim.x + threadIdx.x) * kLagChunk;
  if (i0 >= count) return;
  const uint32_t cnt = min(kLagChunk, count - i0);
  FrEl acc = Fr::one();
  for (uint32_t k = 0; k < cnt; k++) {
    st_vec(out + i0 + k, acc);
    acc = fmul(acc, fsub(tau, pow_from_tables(wlo, whi, i0 + k)));   // non-zero: tau^n != 1
  }
  FrEl inv = Fr::reduce(Fr::inv(acc));
  for (uint32_t k = cnt; k-- > 0;) {
    const FrEl wi = pow_from_tables(wlo, whi, i0 + k);
    const FrEl dinv = fmul(inv, ld_vec(out + i0 + k));
    inv = fmul(inv, fsub(tau, wi));
    st_vec(out + i0 + k, fmul(fmul(zn, wi), dinv));
  }
}

// ---- 2. QAP evaluation y[j] = sum_i M[i][j] L_i: a counting sort of the entries by column (histogram, scan,
// scatter of the products), then a segmented sum over fixed tiles.  Column lengths are extremely skewed (one column
// can hold a sixth of all entries), so no thread owns a column: a thread owns kSegTile consecutive entries, writes the
// columns that begin and end inside its tile, and carries its first and last run to the next level's list (two slots
// per tile), which is reduced the same way until one tile holds it.  Field addition is exact: the scatter order does
// not change the result.
constexpr uint32_t kSegTile = 32;
constexpr uint32_t kNoColumn = 0xffffffffu;
constexpr uint32_t kScanTile = 1024;

__global__ void qap_histogram_kernel(const uint32_t* __restrict__ cols, uint32_t nnz, uint32_t* hist) {
  const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k < nnz) atomicAdd(hist + cols[k], 1u);
}

// exclusive scan in tiles of kScanTile: per-tile sums, one block scans them, every tile applies its offset
__global__ void __launch_bounds__(kScanTile) qap_scan_tiles_kernel(const uint32_t* in, uint32_t count, uint32_t* out,
                                                                   uint32_t* tile_sums) {
  __shared__ uint32_t sh[kScanTile];
  const uint32_t i = blockIdx.x * kScanTile + threadIdx.x;
  const uint32_t v = i < count ? in[i] : 0u;
  sh[threadIdx.x] = v;
  __syncthreads();
  for (uint32_t d = 1; d < kScanTile; d <<= 1) {   // Hillis-Steele, inclusive
    const uint32_t t = threadIdx.x >= d ? sh[threadIdx.x - d] : 0u;
    __syncthreads();
    sh[threadIdx.x] += t;
    __syncthreads();
  }
  if (i < count) out[i] = sh[threadIdx.x] - v;
  if (threadIdx.x == kScanTile - 1) tile_sums[blockIdx.x] = sh[kScanTile - 1];
}
__global__ void qap_scan_sums_kernel(uint32_t* tile_sums, uint32_t ntiles) {   // one thread: ntiles <= 2^16
  if (blockIdx.x != 0 || threadIdx.x != 0) return;
  uint32_t acc = 0;
  for (uint32_t t = 0; t < ntiles; t++) {
    const uint32_t v = tile_sums[t];
    tile_sums[t] = acc;
    acc += v;
  }
}
__global__ void qap_scan_apply_kernel(uint32_t* out, uint32_t count, const uint32_t* tile_sums, uint32_t* cursor) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  const uint32_t v = out[i] + tile_sums[i / kScanTile];
  out[i] = v;
  cursor[i] = v;
}

// entry k of row i (found by binary search in row_ptr) -> its column's next slot, with the product M[i][j] L_i
__global__ void qap_scatter_kernel(const uint32_t* __restrict__ row_ptr, uint32_t nrows, const uint32_t* __restrict__ cols,
                                   const FrEl* __restrict__ coeffs, uint32_t nnz, const FrEl* __restrict__ lag,
                                   uint32_t* cursor, uint32_t* keys, FrEl* vals) {
  const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= nnz) return;
  uint32_t lo = 0, hi = nrows;   // the row i with row_ptr[i] <= k < row_ptr[i + 1]
  while (hi - lo > 1) {
    const uint32_t mid = (lo + hi) >> 1;
    if (row_ptr[mid] <= k) lo = mid;
    else hi = mid;
  }
  const uint32_t j = cols[k];
  const uint32_t pos = atomicAdd(cursor + j, 1u);
  keys[pos] = j;
  st_vec(vals + pos, fmul(Fr::reduce(ld_vec(coeffs + k)), ld_vec(lag + lo)));
}

// one level of the segmented sum: `last` = the list fits in one tile, every run is written
__global__ void __launch_bounds__(128)
    qap_segsum_kernel(const uint32_t* __restrict__ keys, const FrEl* __restrict__ vals, uint32_t count, bool last,
                      uint32_t* next_keys, FrEl* next_vals, FrEl* y) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  const uint32_t begin = t * kSegTile;
  if (begin >= count) return;
  const uint32_t end = min(begin + kSegTile, count);
  uint32_t run_key = kNoColumn, first_key = kNoColumn;
  FrEl acc = Fr::zero(), first = Fr::zero();
  bool have_first = false;
  for (uint32_t k = begin; k < end; k++) {
    const uint32_t key = keys[k];
    if (key == kNoColumn) continue;
    if (key != run_key) {
      if (run_key != kNoColumn) {          // a run closes before the tile's last run
        if (!have_first && !last) {
          first_key = run_key; first = acc; have_first = true;
        } else {
          st_vec(y + run_key, acc);
        }
      }
      run_key = key;
      acc = Fr::zero();
    }
    acc = fadd(acc, ld_vec(vals + k));
  }
  if (last) {
    if (run_key != kNoColumn) st_vec(y + run_key, acc);
    return;
  }
  // carried: the first run (if another one follows) and the last run
  next_keys[2 * t] = have_first ? first_key : run_key;
  st_vec(next_vals + 2 * t, have_first ? first : acc);
  next_keys[2 * t + 1] = have_first ? run_key : kNoColumn;
  st_vec(next_vals + 2 * t + 1, have_first ? acc : Fr::zero());
}

void qap_eval(Ctx& c, const CsrDev& M, uint32_t nrows, uint32_t ncols, const FrEl* lag, FrEl* y, cudaStream_t st) {
  B2Z_CUDA(cudaMemsetAsync(y, 0, (size_t)ncols * sizeof(FrEl), st));
  uint32_t nnz = 0;
  B2Z_CUDA(cudaMemcpyAsync(&nnz, M.row_ptr.p + nrows, 4, cudaMemcpyDeviceToHost, st));
  B2Z_CUDA(cudaStreamSynchronize(st));
  if (nnz == 0) return;
  const uint32_t ntiles = (ncols + kScanTile - 1) / kScanTile;
  DevBuf<uint32_t> hist(ncols), offs(ncols), cursor(ncols), tile_sums(ntiles);
  B2Z_CUDA(cudaMemsetAsync(hist.p, 0, (size_t)ncols * 4, st));
  qap_histogram_kernel<<<nblocks(nnz, 256), 256, 0, st>>>(M.cols.p, nnz, hist.p);
  B2Z_LAUNCHED(&c);
  qap_scan_tiles_kernel<<<ntiles, kScanTile, 0, st>>>(hist.p, ncols, offs.p, tile_sums.p);
  B2Z_LAUNCHED(&c);
  qap_scan_sums_kernel<<<1, 32, 0, st>>>(tile_sums.p, ntiles);
  B2Z_LAUNCHED(&c);
  qap_scan_apply_kernel<<<nblocks(ncols, 256), 256, 0, st>>>(offs.p, ncols, tile_sums.p, cursor.p);
  B2Z_LAUNCHED(&c);
  const uint32_t cap2 = 2 * ((nnz + kSegTile - 1) / kSegTile);
  DevBuf<uint32_t> keys[2] = {DevBuf<uint32_t>(nnz), DevBuf<uint32_t>(cap2)};
  DevBuf<FrEl> vals[2] = {DevBuf<FrEl>(nnz), DevBuf<FrEl>(cap2)};
  qap_scatter_kernel<<<nblocks(nnz, 256), 256, 0, st>>>(M.row_ptr.p, nrows, M.cols.p, M.coeffs.p, nnz, lag, cursor.p,
                                                         keys[0].p, vals[0].p);
  B2Z_LAUNCHED(&c);
  // level k reads list k & 1; a list of count entries leaves 2 ceil(count / kSegTile), which fits the other buffer
  uint32_t count = nnz;
  for (int lvl = 0;; lvl++) {
    const bool last = count <= kSegTile;
    const int in = lvl & 1;
    qap_segsum_kernel<<<nblocks((count + kSegTile - 1) / kSegTile, 128), 128, 0, st>>>(
        keys[in].p, vals[in].p, count, last, keys[in ^ 1].p, vals[in ^ 1].p, y);
    B2Z_LAUNCHED(&c);
    if (last) break;
    count = 2 * ((count + kSegTile - 1) / kSegTile);
  }
  B2Z_CUDA(cudaStreamSynchronize(st));   // the scratch is freed on return
}

// ---- 3. scalars of the variable queries, as canonical integers:
//   a[j] = A_j (+ L_{nc+j}),  b[j] = B_j,  abc = beta A_j + alpha B_j + C_j -> l[j - l] = abc / delta or g[j] = abc / gamma
__global__ void setup_scalars_kernel(const FrEl* __restrict__ qa, const FrEl* __restrict__ qb,
                                     const FrEl* __restrict__ qc, const FrEl* __restrict__ lag_inst, uint32_t m,
                                     uint32_t l, const FrEl alpha, const FrEl beta, const FrEl ginv, const FrEl dinv,
                                     FrEl* sa, FrEl* sb, FrEl* sl, FrEl* sg) {
  const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= m) return;
  FrEl a = ld_vec(qa + j);
  if (j < l) a = fadd(a, ld_vec(lag_inst + j));
  const FrEl b = ld_vec(qb + j);
  st_vec(sa + j, Fr::from_mont(a));
  st_vec(sb + j, Fr::from_mont(b));
  const FrEl abc = fadd(fadd(fmul(beta, a), fmul(alpha, b)), ld_vec(qc + j));
  if (j < l) st_vec(sg + j, Fr::from_mont(fmul(abc, ginv)));
  else st_vec(sl + j - l, Fr::from_mont(fmul(abc, dinv)));
}

// h scalars tau^i Z(tau)/delta (i < n - 1) at bit-reversed position p = bitrev(i) of the n-padded H set; position
// bitrev(n - 1) = n - 1 gets 0, whose multiple is the flagged identity the prover's padding expects
__global__ void setup_h_scalars_kernel(const FrEl* __restrict__ tlo, const FrEl* __restrict__ thi, const FrEl scale,
                                       uint32_t log_n, FrEl* sh) {
  const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= (1u << log_n)) return;
  const uint32_t i = log_n == 0 ? 0 : (__brev(p) >> (32 - log_n));
  st_vec(sh + p, i + 1 < (1u << log_n) ? Fr::from_mont(fmul(scale, pow_from_tables(tlo, thi, i))) : Fr::zero());
}

// ---- host side (hostfr::Fr: 4 x u64 Montgomery limbs, the layout of FrEl)
FrEl dev_el(const hostfr::Fr& x) {
  FrEl e;
  std::memcpy(e.l, x.l, 32);
  return e;
}
hostfr::Fr host_el(const uint64_t* v) { return hostfr::fr_load(v); }

bool g1_on_curve(const host::Fq& x, const host::Fq& y) {   // y^2 = x^3 + 4
  using namespace host;
  return fq_eq(fq_sqr(y), fq_add(fq_mul(fq_sqr(x), x), fq_from_u64(4)));
}
bool g2_on_curve(const host::Fq2& x, const host::Fq2& y) {   // y^2 = x^3 + 4 (1 + u)
  using namespace host;
  const host::Fq four = fq_from_u64(4);
  return fq2_eq(fq2_sqr(y), fq2_add(fq2_mul(fq2_sqr(x), x), host::Fq2{four, four}));
}
bool limbs_zero(const uint64_t* v, int n) {
  uint64_t z = 0;
  for (int i = 0; i < n; i++) z |= v[i];
  return z == 0;
}
bool fq_limbs_canonical(const uint64_t* v, int nfq) {
  for (int k = 0; k < nfq; k++)
    if (host::fq_geq_q(v + 6 * k)) return false;
  return true;
}
void check_g1_generator(const uint64_t* g) {
  B2Z_REQUIRE(!limbs_zero(g, 12), B2Z_EINVAL, "b2z_groth16_setup: g1_generator is the identity");
  B2Z_REQUIRE(fq_limbs_canonical(g, 2), B2Z_EINVAL, "b2z_groth16_setup: g1_generator coordinate not below q");
  host::G1Aff p;
  std::memcpy(p.x.l, g, 48);
  std::memcpy(p.y.l, g + 6, 48);
  p.inf = false;
  B2Z_REQUIRE(g1_on_curve(p.x, p.y), B2Z_EINVAL, "b2z_groth16_setup: g1_generator is not on the curve");
  B2Z_REQUIRE(host::g1_in_subgroup(p), B2Z_EINVAL, "b2z_groth16_setup: g1_generator is not in the r-order subgroup");
}
void check_g2_generator(const uint64_t* g) {
  B2Z_REQUIRE(!limbs_zero(g, 24), B2Z_EINVAL, "b2z_groth16_setup: g2_generator is the identity");
  B2Z_REQUIRE(fq_limbs_canonical(g, 4), B2Z_EINVAL, "b2z_groth16_setup: g2_generator coordinate not below q");
  host::G2Aff p;
  std::memcpy(&p.x, g, 96);
  std::memcpy(&p.y, g + 12, 96);
  p.inf = false;
  B2Z_REQUIRE(g2_on_curve(p.x, p.y), B2Z_EINVAL, "b2z_groth16_setup: g2_generator is not on the curve");
  B2Z_REQUIRE(host::g2_in_subgroup(p), B2Z_EINVAL, "b2z_groth16_setup: g2_generator is not in the r-order subgroup");
}

// x^k for k < count as the tables lo (1024 entries) and hi (ceil(count / 1024) entries)
void pow_tables(Ctx& c, const hostfr::Fr& x, uint32_t count, DevBuf<FrEl>& lo, DevBuf<FrEl>& hi, cudaStream_t st) {
  const uint32_t nhi = (count + 1023) / 1024;
  lo.alloc(1024);
  hi.alloc(nhi ? nhi : 1);
  fr_pow_table(&c, lo.p, dev_el(x), 1024, st);
  fr_pow_table(&c, hi.p, dev_el(hostfr::fr_pow_u64(x, 1024)), nhi ? nhi : 1, st);
}

void groth16_setup(Ctx& c, b2z_r1cs* r1cs, const b2z_setup_desc* d, b2z_pk** pk_out, b2z_vk_out* vk) {
  using namespace hostfr;   // fr_* host arithmetic
  B2Z_REQUIRE(d != nullptr && pk_out != nullptr && vk != nullptr, B2Z_EINVAL, "b2z_groth16_setup: NULL argument");
  B2Z_REQUIRE(d->alpha && d->beta && d->gamma && d->delta && d->tau, B2Z_EINVAL,
              "b2z_groth16_setup: NULL toxic-waste element");
  B2Z_REQUIRE(vk->gamma_abc_g1 && vk->gamma_abc_inf, B2Z_EINVAL, "b2z_groth16_setup: NULL vk_out array");
  const R1csView R = r1cs_view(c, r1cs, "b2z_groth16_setup");
  const uint64_t nc = R.nc, l = R.l, m = R.m;
  const uint32_t log_n = R.log_n;
  B2Z_REQUIRE(log_n <= 26, B2Z_ENOMEM, "b2z_groth16_setup: domain does not fit this build's single-GPU plan");
  B2Z_REQUIRE(m < (1ull << 26), B2Z_ESIZE, "b2z_groth16_setup: too many variables");
  const char* names[5] = {"alpha", "beta", "gamma", "delta", "tau"};
  const uint64_t* els[5] = {d->alpha, d->beta, d->gamma, d->delta, d->tau};
  for (int k = 0; k < 5; k++)
    B2Z_REQUIRE(fr_is_canonical(els[k]), B2Z_EINVAL, std::string("b2z_groth16_setup: ") + names[k] + " is not below r");
  const hostfr::Fr alpha = host_el(d->alpha), beta = host_el(d->beta), gamma = host_el(d->gamma),
                   delta = host_el(d->delta), tau = host_el(d->tau);
  B2Z_REQUIRE(!fr_is_zero(gamma), B2Z_EINVAL, "b2z_groth16_setup: gamma is zero (it has no inverse)");
  B2Z_REQUIRE(!fr_is_zero(delta), B2Z_EINVAL, "b2z_groth16_setup: delta is zero (it has no inverse)");
  const uint64_t n = 1ull << log_n;
  hostfr::Fr tn = tau;
  for (uint32_t i = 0; i < log_n; i++) tn = fr_mul(tn, tn);
  const hostfr::Fr zt = fr_sub(tn, fr_one());   // Z(tau) = tau^n - 1
  B2Z_REQUIRE(!fr_is_zero(zt), B2Z_EINVAL, "b2z_groth16_setup: tau lies in the evaluation domain (tau^n = 1)");
  if (d->g1_generator) check_g1_generator(d->g1_generator);
  if (d->g2_generator) check_g2_generator(d->g2_generator);

  const bool pre = pk_precompute_fits(log_n, m, l);   // before this call's own allocations, as b2z_pk_upload decides
  cudaStream_t st = c.stream;
  const uint32_t nl = (uint32_t)(nc + l);
  hostfr::Fr w = fr_two_adic_root();
  for (uint32_t i = log_n; i < 32; i++) w = fr_mul(w, w);
  const hostfr::Fr dinv = fr_inv(delta), ginv = fr_inv(gamma);

  // 1. Lagrange coefficients
  DevBuf<FrEl> lag(nl);
  {
    DevBuf<FrEl> wlo, whi;
    pow_tables(c, w, nl, wlo, whi, st);
    const hostfr::Fr zn = fr_mul(zt, fr_inv(fr_from_u64(n)));
    setup_lagrange_kernel<<<nblocks(nblocks(nl, kLagChunk), 128), 128, 0, st>>>(wlo.p, whi.p, dev_el(tau),
                                                                                 dev_el(zn), nl, lag.p);
    B2Z_LAUNCHED(&c);
    B2Z_CUDA(cudaStreamSynchronize(st));
  }
  // 2. QAP evaluation
  DevBuf<FrEl> q[3] = {DevBuf<FrEl>(m), DevBuf<FrEl>(m), DevBuf<FrEl>(m)};
  for (int k = 0; k < 3; k++) qap_eval(c, R.mat[k], (uint32_t)nc, (uint32_t)m, lag.p, q[k].p, st);
  // 3. scalars; the set tails (alpha delta | beta delta | delta) as canonical integers from the host
  DevBuf<FrEl> sa(m + 2), sb(m + 2), sl(m - l + 1), sg(l), sh(n), sgamma(1);
  setup_scalars_kernel<<<nblocks(m, 128), 128, 0, st>>>(q[0].p, q[1].p, q[2].p, lag.p + nc, (uint32_t)m, (uint32_t)l,
                                                         dev_el(alpha), dev_el(beta), dev_el(ginv), dev_el(dinv), sa.p,
                                                         sb.p, sl.p, sg.p);
  B2Z_LAUNCHED(&c);
  const hostfr::Fr tails[6] = {fr_into_bigint(alpha), fr_into_bigint(delta), fr_into_bigint(beta),
                               fr_into_bigint(delta), fr_into_bigint(gamma), fr_into_bigint(delta)};
  B2Z_CUDA(cudaMemcpyAsync(sa.p + m, &tails[0], 64, cudaMemcpyHostToDevice, st));
  B2Z_CUDA(cudaMemcpyAsync(sb.p + m, &tails[2], 64, cudaMemcpyHostToDevice, st));
  B2Z_CUDA(cudaMemcpyAsync(sl.p + (m - l), &tails[5], 32, cudaMemcpyHostToDevice, st));
  B2Z_CUDA(cudaMemcpyAsync(sgamma.p, &tails[4], 32, cudaMemcpyHostToDevice, st));
  {
    DevBuf<FrEl> tlo, thi;
    pow_tables(c, tau, (uint32_t)n, tlo, thi, st);
    setup_h_scalars_kernel<<<nblocks(n, 128), 128, 0, st>>>(tlo.p, thi.p, dev_el(fr_mul(zt, dinv)), log_n, sh.p);
    B2Z_LAUNCHED(&c);
    B2Z_CUDA(cudaStreamSynchronize(st));
  }
  lag.release();
  for (auto& v : q) v.release();

  // 4. fixed-base multiplications with the caller's generators (a table of their own) or the standard ones (cached)
  FbTable<G1> own1;
  FbTable<G2> own2;
  if (d->g1_generator) {
    G1::Affine g;
    std::memcpy(&g, d->g1_generator, sizeof(g));
    fb_build<G1>(&c, own1, g, st);
  }
  if (d->g2_generator) {
    G2::Affine g;
    std::memcpy(&g, d->g2_generator, sizeof(g));
    fb_build<G2>(&c, own2, g, st);
  }
  const FbTable<G1>& t1 = d->g1_generator ? own1 : fb_standard_table<G1>(&c, st);
  const FbTable<G2>& t2 = d->g2_generator ? own2 : fb_standard_table<G2>(&c, st);
  auto words = [](uint64_t count) { return DevBuf<uint32_t>((count + 31) / 32 + 1); };
  DevBuf<G1::Affine> pa(m + 2), pb1(m + 2), pl(m - l + 1), ph(n), pg(l);
  DevBuf<G2::Affine> pb2(m + 2), pgamma(1);
  DevBuf<uint32_t> wa = words(m + 2), wb1 = words(m + 2), wl = words(m - l + 1), wh = words(n), wg = words(l),
                   wb2 = words(m + 2), wgamma = words(1);
  fixed_base_mul<G1>(&c, t1, sa.p, pa.p, wa.p, (uint32_t)m + 2, st);
  fixed_base_mul<G1>(&c, t1, sb.p, pb1.p, wb1.p, (uint32_t)m + 2, st);
  fixed_base_mul<G1>(&c, t1, sl.p, pl.p, wl.p, (uint32_t)(m - l) + 1, st);
  fixed_base_mul<G1>(&c, t1, sh.p, ph.p, wh.p, (uint32_t)n, st);
  fixed_base_mul<G1>(&c, t1, sg.p, pg.p, wg.p, (uint32_t)l, st);
  fixed_base_mul<G2>(&c, t2, sb.p, pb2.p, wb2.p, (uint32_t)m + 2, st);
  fixed_base_mul<G2>(&c, t2, sgamma.p, pgamma.p, wgamma.p, 1, st);

  // 5. verifying key: alpha_1 and beta_2, delta_2 from the set tails, gamma_2, gamma_abc
  std::vector<uint32_t> gw((l + 31) / 32);
  B2Z_CUDA(cudaMemcpyAsync(vk->alpha_g1, pa.p + m, sizeof(G1::Affine), cudaMemcpyDeviceToHost, st));
  B2Z_CUDA(cudaMemcpyAsync(vk->beta_g2, pb2.p + m, sizeof(G2::Affine), cudaMemcpyDeviceToHost, st));
  B2Z_CUDA(cudaMemcpyAsync(vk->delta_g2, pb2.p + m + 1, sizeof(G2::Affine), cudaMemcpyDeviceToHost, st));
  B2Z_CUDA(cudaMemcpyAsync(vk->gamma_g2, pgamma.p, sizeof(G2::Affine), cudaMemcpyDeviceToHost, st));
  B2Z_CUDA(cudaMemcpyAsync(vk->gamma_abc_g1, pg.p, l * sizeof(G1::Affine), cudaMemcpyDeviceToHost, st));
  B2Z_CUDA(cudaMemcpyAsync(gw.data(), wg.p, gw.size() * 4, cudaMemcpyDeviceToHost, st));
  B2Z_CUDA(cudaStreamSynchronize(st));
  std::memcpy(vk->gamma_abc_inf, gw.data(), (l + 7) / 8);

  // 6. the key, assembled as b2z_pk_upload assembles it
  const PkDeviceSets sets{pa.p, pb1.p, pl.p, ph.p, pb2.p, wa.p, wb1.p, wl.p, wh.p, wb2.p};
  *pk_out = pk_from_device_sets(c, log_n, m, l, sets, pre);
}

}  // namespace
}  // namespace b2z

extern "C" b2z_status b2z_groth16_setup(b2z_ctx* ctx, b2z_r1cs* r1cs, const b2z_setup_desc* desc, b2z_pk** pk_out,
                                        b2z_vk_out* vk_out) {
  if (pk_out) *pk_out = nullptr;
  return b2z::guarded(ctx, [&](b2z::Ctx& c) { b2z::groth16_setup(c, r1cs, desc, pk_out, vk_out); });
}
