// Constraint-row evaluation on the device -- the `evaluate_constraint` loop at the top of
// ark-groth16's LibsnarkReduction::witness_map_from_matrices (SURVEY.md A.3, row a3/f1):
//   a[i] = <A_i, z>, b[i] = <B_i, z>, c[i] = <C_i, z>   for i < num_constraints
//   a[num_constraints + j] = z[j]                       for j < num_instance ; zero elsewhere
// The matrices are static per circuit: uploaded once as CSR (row offsets, column indices,
// Montgomery coefficients), then every proof sends only z (32 B per variable) instead of the
// three evaluation vectors (96 B per domain point).  A gather-bound kernel: one thread per row.
#include <algorithm>
#include <cstring>
#include <vector>

#include "api_glue.hpp"
#include "msm.hpp"
#include "prove_internal.hpp"

namespace b2z {

// Two-pass row evaluation.  The rows of these circuits are wildly uneven (1 entry for a multiplication gate, up to
// 33 for an inlined Poseidon MDS row; a warp of 32 consecutive rows does 3.3x the multiplications it needs when one
// thread owns one row), so the multiplications are done per ENTRY (perfectly balanced; entries whose coefficient is
// 1 -- every multiplication-gate row -- are plain copies, flagged in the column word) and only the cheap additions
// per row.  `rows_out` outputs per matrix; the instance rows a[nc + j] = z[j] are ordinary one-entry rows of A.
constexpr uint32_t kCoefOne = 0x80000000u;
struct EvalPlan {
  DevBuf<uint32_t> rp[3], ci[3];
  DevBuf<FrEl> cf[3];
  DevBuf<FrEl> prod;               // the three matrices' products back to back
  uint32_t nnz[3] = {0, 0, 0};
  uint32_t rows_out = 0;
};

struct R1csImpl {
  const Ctx* owner = nullptr;      // holds per-proof scratch (z, ea, eb, ec): belongs to the uploading context
  EvalPlan plan;                   // all n rows, natural order
  uint64_t nc = 0, l = 0, m = 0;
  uint32_t log_n = 0;
  CsrDev mat[3];
  DevBuf<FrEl> z, ea, eb, ec;
  cudaEvent_t ev_z = nullptr;      // z uploaded (b2z_groth16_shard_begin / b2z_r1cs_coset_evals, whichever came first)
  bool z_valid = false;
  ~R1csImpl() {
    if (ev_z) cudaEventDestroy(ev_z);
  }
};

namespace {

__device__ __forceinline__ FrEl ldg32(const FrEl* p) {
  const uint4* q = reinterpret_cast<const uint4*>(p);
  const uint4 a = __ldg(q), b = __ldg(q + 1);
  FrEl r;
  r.l[0] = a.x; r.l[1] = a.y; r.l[2] = a.z; r.l[3] = a.w;
  r.l[4] = b.x; r.l[5] = b.y; r.l[6] = b.z; r.l[7] = b.w;
  return r;
}

__device__ __forceinline__ FrEl ld32(const FrEl* p) {
  const uint4* q = reinterpret_cast<const uint4*>(p);
  const uint4 a = q[0], b = q[1];
  FrEl r;
  r.l[0] = a.x; r.l[1] = a.y; r.l[2] = a.z; r.l[3] = a.w;
  r.l[4] = b.x; r.l[5] = b.y; r.l[6] = b.z; r.l[7] = b.w;
  return r;
}

// y = M x  for a CSR matrix over Fr (x, coefficients canonical Montgomery); one thread per row
__global__ void spmv_kernel(const uint32_t* __restrict__ rp, const uint32_t* __restrict__ ci,
                            const FrEl* __restrict__ cf, const FrEl* __restrict__ x, uint32_t nrows, FrEl* y) {
  const uint32_t row = blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= nrows) return;
  FrEl acc = Fr::zero();
  const uint32_t end = rp[row + 1];
  for (uint32_t k = rp[row]; k < end; k++) acc = Fr::add(acc, Fr::mul(ldg32(cf + k), ldg32(x + ci[k])));
  y[row] = Fr::reduce(acc);
}

__global__ void r1cs_products_kernel(const uint32_t* __restrict__ ci0, const FrEl* __restrict__ cf0, uint32_t n0,
                                     const uint32_t* __restrict__ ci1, const FrEl* __restrict__ cf1, uint32_t n1,
                                     const uint32_t* __restrict__ ci2, const FrEl* __restrict__ cf2, uint32_t n2,
                                     const FrEl* __restrict__ z, FrEl* prod) {
  const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
  const uint32_t which = blockIdx.y;
  const uint32_t cnt = which == 0 ? n0 : (which == 1 ? n1 : n2);
  if (k >= cnt) return;
  const uint32_t* ci = which == 0 ? ci0 : (which == 1 ? ci1 : ci2);
  const FrEl* cf = which == 0 ? cf0 : (which == 1 ? cf1 : cf2);
  FrEl* out = prod + (which == 0 ? 0 : (which == 1 ? n0 : n0 + n1));
  const uint32_t c = ci[k];
  const FrEl zv = ldg32(z + (c & ~kCoefOne));
  out[k] = (c & kCoefOne) ? zv : Fr::mul(ldg32(cf + k), zv);   // coefficient canonical, result lazy
}

__global__ void r1cs_rowsum_kernel(const uint32_t* __restrict__ rp0, const uint32_t* __restrict__ rp1,
                                   const uint32_t* __restrict__ rp2, uint32_t n0, uint32_t n1,
                                   const FrEl* __restrict__ prod, uint32_t rows, FrEl* a, FrEl* b, FrEl* c) {
  const uint32_t row = blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= rows) return;
  const uint32_t which = blockIdx.y;
  const uint32_t* rp = which == 0 ? rp0 : (which == 1 ? rp1 : rp2);
  const FrEl* p = prod + (which == 0 ? 0 : (which == 1 ? n0 : n0 + n1));
  FrEl* out = which == 0 ? a : (which == 1 ? b : c);
  FrEl acc = Fr::zero();
  const uint32_t end = rp[row + 1];
  for (uint32_t k = rp[row]; k < end; k++) acc = Fr::add(acc, ld32(p + k));
  out[row] = Fr::reduce(acc);
}

// Host CSR of one matrix (as uploaded) -> the plan's arrays for `rows_out` outputs, output row j being global row
// row_of(j) (>= nc + extra: empty).  Matrix A carries the l instance rows after its nc constraint rows.
struct HostCsr {
  std::vector<uint32_t> rp, ci;
  std::vector<FrEl> cf;
};
template <class RowOf>
void plan_matrix(EvalPlan& P, int k, const HostCsr& M, uint64_t nc, uint64_t l, uint32_t rows_out, RowOf row_of,
                 cudaStream_t st) {
  const FrEl one = Fr::one();
  std::vector<uint32_t> rp(rows_out + 1, 0), ci;
  std::vector<FrEl> cf;
  for (uint32_t j = 0; j < rows_out; j++) {
    const uint64_t row = row_of(j);
    if (row < nc) {
      for (uint32_t e = M.rp[row]; e < M.rp[row + 1]; e++) {
        const bool is_one = std::memcmp(M.cf[e].l, one.l, sizeof(one.l)) == 0;
        ci.push_back(M.ci[e] | (is_one ? kCoefOne : 0u));
        cf.push_back(M.cf[e]);
      }
    } else if (k == 0 && row < nc + l) {
      ci.push_back((uint32_t)(row - nc) | kCoefOne);
      cf.push_back(one);
    }
    rp[j + 1] = (uint32_t)ci.size();
  }
  P.nnz[k] = (uint32_t)ci.size();
  P.rp[k].alloc(rp.size());
  P.ci[k].alloc(ci.size() ? ci.size() : 1);
  P.cf[k].alloc(cf.size() ? cf.size() : 1);
  B2Z_CUDA(cudaMemcpyAsync(P.rp[k].p, rp.data(), rp.size() * 4, cudaMemcpyHostToDevice, st));
  if (!ci.empty()) {
    B2Z_CUDA(cudaMemcpyAsync(P.ci[k].p, ci.data(), ci.size() * 4, cudaMemcpyHostToDevice, st));
    B2Z_CUDA(cudaMemcpyAsync(P.cf[k].p, cf.data(), cf.size() * sizeof(FrEl), cudaMemcpyHostToDevice, st));
  }
  B2Z_CUDA(cudaStreamSynchronize(st));   // the vectors are locals
}
void plan_finish(EvalPlan& P, uint32_t rows_out) {
  P.rows_out = rows_out;
  const size_t total = (size_t)P.nnz[0] + P.nnz[1] + P.nnz[2];
  P.prod.alloc(total ? total : 1);
}
// device CSR -> host (dist set-up: the caller's arrays are gone by then)
HostCsr download_csr(const CsrDev& d, uint64_t nc, cudaStream_t st) {
  HostCsr h;
  h.rp.resize(nc + 1);
  B2Z_CUDA(cudaMemcpyAsync(h.rp.data(), d.row_ptr.p, (nc + 1) * 4, cudaMemcpyDeviceToHost, st));
  B2Z_CUDA(cudaStreamSynchronize(st));
  const size_t nnz = h.rp[nc];
  h.ci.resize(nnz);
  h.cf.resize(nnz);
  if (nnz) {
    B2Z_CUDA(cudaMemcpyAsync(h.ci.data(), d.cols.p, nnz * 4, cudaMemcpyDeviceToHost, st));
    B2Z_CUDA(cudaMemcpyAsync(h.cf.data(), d.coeffs.p, nnz * sizeof(FrEl), cudaMemcpyDeviceToHost, st));
    B2Z_CUDA(cudaStreamSynchronize(st));
  }
  return h;
}
void run_plan(Ctx& c, const EvalPlan& P, const FrEl* d_z, FrEl* a, FrEl* b, FrEl* cc, cudaStream_t st) {
  ProfileScope ps(&c, PH_R1CS_EVAL, st, 3ull * P.rows_out);
  const uint32_t mx = std::max(P.nnz[0], std::max(P.nnz[1], P.nnz[2]));
  if (mx) {
    r1cs_products_kernel<<<dim3((mx + 255) / 256, 3), 256, 0, st>>>(P.ci[0].p, P.cf[0].p, P.nnz[0], P.ci[1].p, P.cf[1].p,
                                                                   P.nnz[1], P.ci[2].p, P.cf[2].p, P.nnz[2], d_z, P.prod.p);
    B2Z_LAUNCHED(&c);
  }
  r1cs_rowsum_kernel<<<dim3((P.rows_out + 255) / 256, 3), 256, 0, st>>>(P.rp[0].p, P.rp[1].p, P.rp[2].p, P.nnz[0], P.nnz[1],
                                                                       P.prod.p, P.rows_out, a, b, cc);
  B2Z_LAUNCHED(&c);
}

// This rank's slice of the assignment -> the same offsets of every peer's buffer, by NVLink stores (one launch;
// seven peer copies through the copy engines cost ~0.2 ms each with IPC-mapped destinations).
struct PeerPtrs {
  uint4* p[8];
};
__global__ void z_scatter_kernel(const uint4* __restrict__ src, size_t count16, PeerPtrs dst, uint32_t npeers) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < count16; i += stride) {
    const uint4 v = src[i];
    for (uint32_t k = 0; k < npeers; k++) dst.p[k][i] = v;
  }
}

void upload_csr(CsrDev& d, const uint64_t* row_ptr, const uint32_t* cols, const uint64_t* coeffs, uint64_t nc,
                uint64_t m, cudaStream_t st) {
  B2Z_REQUIRE(row_ptr != nullptr, B2Z_EINVAL, "b2z_r1cs_upload: NULL row_ptr");
  const uint64_t nnz = row_ptr[nc];
  B2Z_REQUIRE(row_ptr[0] == 0 && nnz < (1ull << 32), B2Z_EINVAL, "b2z_r1cs_upload: bad row_ptr");
  B2Z_REQUIRE(nnz == 0 || (cols != nullptr && coeffs != nullptr), B2Z_EINVAL, "b2z_r1cs_upload: NULL entries");
  std::vector<uint32_t> rp(nc + 1);
  for (uint64_t i = 0; i <= nc; i++) {
    B2Z_REQUIRE(i == 0 || row_ptr[i] >= row_ptr[i - 1], B2Z_EINVAL, "b2z_r1cs_upload: row_ptr not monotone");
    rp[i] = (uint32_t)row_ptr[i];
  }
  for (uint64_t k = 0; k < nnz; k++) B2Z_REQUIRE(cols[k] < m, B2Z_EINVAL, "b2z_r1cs_upload: column out of range");
  d.row_ptr.alloc(nc + 1);
  d.cols.alloc(nnz ? nnz : 1);
  d.coeffs.alloc(nnz ? nnz : 1);
  B2Z_CUDA(cudaMemcpyAsync(d.row_ptr.p, rp.data(), (nc + 1) * 4, cudaMemcpyHostToDevice, st));
  if (nnz) {
    B2Z_CUDA(cudaMemcpyAsync(d.cols.p, cols, nnz * 4, cudaMemcpyHostToDevice, st));
    B2Z_CUDA(cudaMemcpyAsync(d.coeffs.p, coeffs, nnz * sizeof(FrEl), cudaMemcpyHostToDevice, st));
  }
  B2Z_CUDA(cudaStreamSynchronize(st));   // rp is a local
}

// rows of ONE matrix (0 = A with the instance rows appended, 1 = B, 2 = C) against z, zero-padded to the domain
void eval_one(Ctx& c, R1csImpl& R, uint32_t which, const FrEl* d_z, FrEl* out, cudaStream_t st) {
  const size_t n = (size_t)1 << R.log_n;
  ProfileScope ps(&c, PH_R1CS_EVAL, st, R.nc + (which == 0 ? R.l : 0));
  B2Z_CUDA(cudaMemsetAsync(out, 0, n * sizeof(FrEl), st));
  if (R.nc) {
    spmv_kernel<<<(uint32_t)((R.nc + 127) / 128), 128, 0, st>>>(R.mat[which].row_ptr.p, R.mat[which].cols.p,
                                                              R.mat[which].coeffs.p, d_z, (uint32_t)R.nc, out);
    B2Z_LAUNCHED(&c);
  }
  if (which == 0) {
    B2Z_CUDA(cudaMemcpyAsync(out + R.nc, d_z, R.l * sizeof(FrEl), cudaMemcpyDeviceToDevice, st));
    fr_canonicalize(&c, out + R.nc, R.l, st);
  }
}

}  // namespace
}  // namespace b2z

using namespace b2z;

struct b2z_r1cs {
  R1csImpl impl;
};

namespace b2z {
namespace {
R1csImpl& r1cs_of(Ctx& c, b2z_r1cs* r, const char* who) {
  if (r == nullptr) throw StatusError{B2Z_EINVAL, std::string(who) + ": r1cs is NULL"};
  if (r->impl.owner != &c)
    throw StatusError{B2Z_EINVAL, std::string(who) + ": this b2z_r1cs was uploaded through another b2z_ctx (a handle "
                                                     "belongs to one context; upload one copy per context)"};
  return r->impl;
}
// the key of a proof on these matrices: uploaded through this context, for a circuit of the same shape
PkImpl& pk_for(Ctx& c, const b2z_pk* pk, const R1csImpl& R, const char* who) {
  PkImpl& P = pk_of(c, pk, who);
  if (P.log_n != R.log_n || P.m != R.m || P.l != R.l)
    throw StatusError{B2Z_EINVAL, std::string(who) + ": key and matrices disagree"};
  return P;
}
// z goes up once, on the stream that prepares the MSM scalars; the row evaluation reads it on the main stream
// after an event.  cudaMemcpyDefault: z may also be a DEVICE pointer (assignment already resident).
void stage_z_and_rows(Ctx& c, R1csImpl& R, const uint64_t* z) {
  B2Z_CUDA(cudaMemcpyAsync(R.z.p, z, R.m * sizeof(FrEl), cudaMemcpyDefault, c.aux[0]));
  B2Z_CUDA(cudaEventRecord(R.ev_z, c.aux[0]));
  B2Z_CUDA(cudaStreamWaitEvent(c.stream, R.ev_z, 0));
  run_plan(c, R.plan, R.z.p, R.ea.p, R.eb.p, R.ec.p, c.stream);
}
}  // namespace
R1csView r1cs_view(Ctx& c, b2z_r1cs* r, const char* who) {
  const R1csImpl& R = r1cs_of(c, r, who);
  return R1csView{R.nc, R.l, R.m, R.log_n, R.mat};
}
}  // namespace b2z

extern "C" {

b2z_status b2z_r1cs_upload(b2z_ctx* ctx, uint64_t num_constraints, uint64_t num_instance, uint64_t num_variables,
                           const uint64_t* a_row_ptr, const uint32_t* a_cols, const uint64_t* a_coeffs,
                           const uint64_t* b_row_ptr, const uint32_t* b_cols, const uint64_t* b_coeffs,
                           const uint64_t* c_row_ptr, const uint32_t* c_cols, const uint64_t* c_coeffs, b2z_r1cs** out) {
  if (out) *out = nullptr;
  return guarded(ctx, [&](Ctx& c) {
    B2Z_REQUIRE(out != nullptr, B2Z_EINVAL, "b2z_r1cs_upload: NULL out");
    B2Z_REQUIRE(num_instance >= 1 && num_variables >= num_instance, B2Z_EINVAL, "b2z_r1cs_upload: bad variable counts");
    uint32_t log_n = 0;
    while ((1ull << log_n) < num_constraints + num_instance) log_n++;
    B2Z_REQUIRE(log_n <= 32, B2Z_ESIZE, "b2z_r1cs_upload: domain larger than 2^32 (PolynomialDegreeTooLarge)");
    B2Z_REQUIRE(log_n <= 28, B2Z_ENOMEM, "b2z_r1cs_upload: domain does not fit this build's single-GPU plan");
    std::unique_ptr<b2z_r1cs> r(new b2z_r1cs());
    R1csImpl& R = r->impl;
    R.owner = &c;
    R.nc = num_constraints; R.l = num_instance; R.m = num_variables; R.log_n = log_n;
    upload_csr(R.mat[0], a_row_ptr, a_cols, a_coeffs, num_constraints, num_variables, c.stream);
    upload_csr(R.mat[1], b_row_ptr, b_cols, b_coeffs, num_constraints, num_variables, c.stream);
    upload_csr(R.mat[2], c_row_ptr, c_cols, c_coeffs, num_constraints, num_variables, c.stream);
    const size_t n = (size_t)1 << log_n;
    {
      const uint64_t* rps[3] = {a_row_ptr, b_row_ptr, c_row_ptr};
      const uint32_t* cis[3] = {a_cols, b_cols, c_cols};
      const uint64_t* cfs[3] = {a_coeffs, b_coeffs, c_coeffs};
      for (int k = 0; k < 3; k++) {
        HostCsr h;
        const uint64_t nnz = rps[k][num_constraints];
        h.rp.resize(num_constraints + 1);
        for (uint64_t i = 0; i <= num_constraints; i++) h.rp[i] = (uint32_t)rps[k][i];
        h.ci.assign(cis[k], cis[k] + nnz);
        h.cf.resize(nnz);
        if (nnz) std::memcpy(h.cf.data(), cfs[k], nnz * sizeof(FrEl));
        plan_matrix(R.plan, k, h, num_constraints, num_instance, (uint32_t)n, [](uint32_t j) { return (uint64_t)j; },
                    c.stream);
      }
      plan_finish(R.plan, (uint32_t)n);
    }
    R.z.alloc(num_variables); R.ea.alloc(n); R.eb.alloc(n); R.ec.alloc(n);
    B2Z_CUDA(cudaEventCreateWithFlags(&R.ev_z, cudaEventDisableTiming));
    *out = r.release();
  });
}

void b2z_r1cs_free(b2z_ctx* ctx, b2z_r1cs* r) {
  if (r == nullptr) return;
  if (ctx != nullptr) {
    std::lock_guard<std::mutex> lock(ctx->impl.mu);
    cudaSetDevice(ctx->impl.device);
    cudaDeviceSynchronize();
  }
  delete r;
}

b2z_status b2z_r1cs_eval(b2z_ctx* ctx, b2z_r1cs* r, const uint64_t* z, uint64_t* a_out, uint64_t* b_out,
                         uint64_t* c_out) {
  return guarded(ctx, [&](Ctx& c) {
    B2Z_REQUIRE(r && z && a_out && b_out && c_out, B2Z_EINVAL, "b2z_r1cs_eval: NULL argument");
    R1csImpl& R = r1cs_of(c, r, "b2z_r1cs_eval");
    const size_t n = (size_t)1 << R.log_n;
    cudaStream_t st = c.stream;
    B2Z_CUDA(cudaMemcpyAsync(R.z.p, z, R.m * sizeof(FrEl), cudaMemcpyHostToDevice, st));
    run_plan(c, R.plan, R.z.p, R.ea.p, R.eb.p, R.ec.p, st);
    B2Z_CUDA(cudaMemcpyAsync(a_out, R.ea.p, n * sizeof(FrEl), cudaMemcpyDeviceToHost, st));
    B2Z_CUDA(cudaMemcpyAsync(b_out, R.eb.p, n * sizeof(FrEl), cudaMemcpyDeviceToHost, st));
    B2Z_CUDA(cudaMemcpyAsync(c_out, R.ec.p, n * sizeof(FrEl), cudaMemcpyDeviceToHost, st));
    B2Z_CUDA(cudaStreamSynchronize(st));
  });
}

b2z_status b2z_spmv_fr(b2z_ctx* ctx, uint64_t nrows, uint64_t ncols, const uint64_t* row_ptr, const uint32_t* cols,
                       const uint64_t* coeffs, const uint64_t* x, uint64_t* y_out) {
  return guarded(ctx, [&](Ctx& c) {
    B2Z_REQUIRE(row_ptr && x && y_out, B2Z_EINVAL, "b2z_spmv_fr: NULL argument");
    B2Z_REQUIRE(nrows < (1ull << 31) && ncols < (1ull << 31), B2Z_ESIZE, "b2z_spmv_fr: matrix too large");
    CsrDev d;
    upload_csr(d, row_ptr, cols, coeffs, nrows, ncols, c.stream);
    DevBuf<FrEl> dx(ncols ? ncols : 1), dy(nrows ? nrows : 1);
    B2Z_CUDA(cudaMemcpyAsync(dx.p, x, ncols * sizeof(FrEl), cudaMemcpyHostToDevice, c.stream));
    if (nrows) {
      spmv_kernel<<<(uint32_t)((nrows + 127) / 128), 128, 0, c.stream>>>(d.row_ptr.p, d.cols.p, d.coeffs.p, dx.p,
                                                                        (uint32_t)nrows, dy.p);
      B2Z_LAUNCHED(&c);
    }
    B2Z_CUDA(cudaMemcpyAsync(y_out, dy.p, nrows * sizeof(FrEl), cudaMemcpyDeviceToHost, c.stream));
    B2Z_CUDA(cudaStreamSynchronize(c.stream));
  });
}

b2z_status b2z_witness_map_from_matrices(b2z_ctx* ctx, b2z_r1cs* r, const uint64_t* z, uint64_t* h_out) {
  return guarded(ctx, [&](Ctx& c) {
    B2Z_REQUIRE(r && z && h_out, B2Z_EINVAL, "b2z_witness_map_from_matrices: NULL argument");
    R1csImpl& R = r1cs_of(c, r, "b2z_witness_map_from_matrices");
    const size_t n = (size_t)1 << R.log_n;
    cudaStream_t st = c.stream;
    B2Z_CUDA(cudaMemcpyAsync(R.z.p, z, R.m * sizeof(FrEl), cudaMemcpyHostToDevice, st));
    run_plan(c, R.plan, R.z.p, R.ea.p, R.eb.p, R.ec.p, st);
    witness_map_device(&c, R.ea.p, R.eb.p, R.ec.p, R.log_n, /*natural_out=*/true, st);
    B2Z_CUDA(cudaMemcpyAsync(h_out, R.ea.p, n * sizeof(FrEl), cudaMemcpyDeviceToHost, st));
    B2Z_CUDA(cudaStreamSynchronize(st));
  });
}

b2z_status b2z_groth16_prove_r1cs(b2z_ctx* ctx, const b2z_pk* pk, b2z_r1cs* r, const uint64_t* z, const uint64_t rr[4],
                                  const uint64_t ss[4], uint8_t proof_out[192]) {
  return guarded(ctx, [&](Ctx& c) {
    B2Z_REQUIRE(pk && r && z && rr && ss && proof_out, B2Z_EINVAL, "b2z_groth16_prove_r1cs: NULL argument");
    R1csImpl& R = r1cs_of(c, r, "b2z_groth16_prove_r1cs");
    PkImpl& P = pk_for(c, pk, R, "b2z_groth16_prove_r1cs");
    stage_z_and_rows(c, R, z);
    prove_device(c, P, R.ea.p, R.eb.p, R.ec.p, R.z.p, rr, ss, proof_out);
  });
}

b2z_status b2z_groth16_prove_partial_r1cs(b2z_ctx* ctx, const b2z_pk* pk, b2z_r1cs* r, const uint64_t* z,
                                          const uint64_t rr[4], const uint64_t ss[4], uint8_t* partial_out) {
  return guarded(ctx, [&](Ctx& c) {
    B2Z_REQUIRE(pk && r && z && rr && ss && partial_out, B2Z_EINVAL, "b2z_groth16_prove_partial_r1cs: NULL argument");
    R1csImpl& R = r1cs_of(c, r, "b2z_groth16_prove_partial_r1cs");
    PkImpl& P = pk_for(c, pk, R, "b2z_groth16_prove_partial_r1cs");
    stage_z_and_rows(c, R, z);
    prove_partial_device(c, P, R.ea.p, R.eb.p, R.ec.p, R.z.p, rr, ss, partial_out);
  });
}

// ---- point-sharded proof with a distributed witness map (include/b200zk.h) ----
namespace {
// z != NULL: upload the assignment (aux stream 0, where the MSM scalars are prepared) and mark it;
// z == NULL: reuse the one uploaded by the previous shard call on this r1cs
void shard_assignment(Ctx& c, R1csImpl& R, const uint64_t* z, const char* who) {
  if (z != nullptr) {
    B2Z_CUDA(cudaMemcpyAsync(R.z.p, z, R.m * sizeof(FrEl), cudaMemcpyDefault, c.aux[0]));
    B2Z_CUDA(cudaEventRecord(R.ev_z, c.aux[0]));
    R.z_valid = true;
  }
  if (!R.z_valid) throw StatusError{B2Z_EINVAL, std::string(who) + ": no assignment uploaded yet (z is NULL)"};
}
}  // namespace

b2z_status b2z_groth16_shard_begin(b2z_ctx* ctx, const b2z_pk* pk, b2z_r1cs* r, const uint64_t* z, const uint64_t rr[4],
                                   const uint64_t ss[4]) {
  return guarded(ctx, [&](Ctx& c) {
    B2Z_REQUIRE(pk && r && rr && ss, B2Z_EINVAL, "b2z_groth16_shard_begin: NULL argument");
    R1csImpl& R = r1cs_of(c, r, "b2z_groth16_shard_begin");
    PkImpl& P = pk_for(c, pk, R, "b2z_groth16_shard_begin");
    shard_assignment(c, R, z, "b2z_groth16_shard_begin");
    B2Z_CUDA(cudaStreamWaitEvent(c.aux[0], R.ev_z, 0));
    proof_begin(c, P, R.z.p, rr, ss);
    proof_accums(c, P, nullptr);
    // the uploaded assignment is valid for THIS proof only: shard_finish clears the flag, so a later call with
    // z == NULL outside a begin/finish window fails instead of silently proving a stale assignment
    P.assignment_flag = &R.z_valid;
  });
}

b2z_status b2z_r1cs_coset_evals(b2z_ctx* ctx, b2z_r1cs* r, uint32_t which, const uint64_t* z, uint64_t* d_out) {
  return guarded(ctx, [&](Ctx& c) {
    B2Z_REQUIRE(r && d_out && which < 3, B2Z_EINVAL, "b2z_r1cs_coset_evals: bad argument");
    R1csImpl& R = r1cs_of(c, r, "b2z_r1cs_coset_evals");
    shard_assignment(c, R, z, "b2z_r1cs_coset_evals");
    cudaStream_t st = c.stream;
    B2Z_CUDA(cudaStreamWaitEvent(st, R.ev_z, 0));
    FrEl* out = reinterpret_cast<FrEl*>(d_out);
    eval_one(c, R, which, R.z.p, out, st);
    witness_map_transform(&c, out, R.log_n, st);
    B2Z_CUDA(cudaStreamSynchronize(st));
  });
}

b2z_status b2z_groth16_shard_finish(b2z_ctx* ctx, const b2z_pk* pk, uint64_t* d_a, const uint64_t* d_b,
                                    const uint64_t* d_c, uint8_t* partial_out) {
  return guarded(ctx, [&](Ctx& c) {
    B2Z_REQUIRE(pk && d_a && d_b && d_c && partial_out, B2Z_EINVAL, "b2z_groth16_shard_finish: NULL argument");
    PkImpl& P = pk_of(c, pk, "b2z_groth16_shard_finish");
    if (P.assignment_flag != nullptr) {
      *P.assignment_flag = false;
      P.assignment_flag = nullptr;
    }
    FrEl* a = reinterpret_cast<FrEl*>(d_a);
    witness_map_quotient(&c, a, reinterpret_cast<const FrEl*>(d_b), reinterpret_cast<const FrEl*>(d_c), P.log_n,
                         /*natural_out=*/false, c.stream);    // whole domain, every shard
    proof_h_sort(c, P, a + P.h_lo, c.stream);
    proof_h_finish(c, P);
    proof_end(c, P, partial_out);
  });
}


// ---- tile-sharded prover: ONE proof by W = 2, 4 or 8 GPUs with the witness map itself distributed ----------------
// (include/b200zk.h, b2z_dist_*).  Data moves by stores / copies into the peers' memory over NVLink; the only
// synchronisation is a host-side barrier on a few words of caller-provided shared host memory.
}  // extern "C"

namespace b2z {
namespace {
constexpr uint32_t kFlagStride = 16;   // u32 words between two ranks' flags (one cache line each)
constexpr size_t kPartial = B2Z_PARTIAL_BYTES;
}  // namespace
struct DistImpl {
  const Ctx* owner = nullptr;
  uint32_t rank = 0, world = 1, wbits = 0, log_n = 0;
  uint64_t m = 0;
  size_t nl = 0, z_bytes = 0, region_bytes = 0;
  PkImpl* pk = nullptr;
  b2z_r1cs* r1cs = nullptr;
  DevBuf<uint8_t> region;                 // [ z (m x 32 B) | X_a X_b X_c | Y_a Y_b Y_c ]  (n / W elements each)
  uint8_t* peer_region[8] = {};
  bool peer_ipc[8] = {};
  uint32_t* flags = nullptr;              // shared host memory: world x kFlagStride u32, then world x 1344 B
  uint8_t* partials = nullptr;
  uint32_t epoch = 0;
  cudaStream_t wm_st = nullptr;
  cudaEvent_t ev_ready = nullptr;
  NttDist nd;
  EvalPlan plan;                          // this rank's rows of the column-owned layout, local order
  ~DistImpl() {
    for (uint32_t p = 0; p < 8; p++)
      if (peer_ipc[p] && peer_region[p]) cudaIpcCloseMemHandle(peer_region[p]);
    if (wm_st) cudaStreamDestroy(wm_st);
    if (ev_ready) cudaEventDestroy(ev_ready);
  }
  FrEl* z() const { return reinterpret_cast<FrEl*>(region.p); }
  uint8_t* vec_of(uint8_t* base, int layout /*0 X, 1 Y*/, int v) const {
    return base + z_bytes + ((size_t)layout * 3 + v) * nl * sizeof(FrEl);
  }
};
namespace {
// host barrier of the ranks on the shared flag words; false = a peer never arrived
bool shared_barrier(uint32_t* flags, uint32_t rank, uint32_t world, uint32_t* epoch) {
  const uint32_t e = ++*epoch;
  __atomic_store_n(flags + rank * kFlagStride, e, __ATOMIC_RELEASE);
  uint64_t spins = 0;
  for (uint32_t p = 0; p < world; p++) {
    // wrap-safe: the peer's epoch has reached ours
    while ((int32_t)(__atomic_load_n(flags + p * kFlagStride, __ATOMIC_ACQUIRE) - e) < 0) {
#if defined(__x86_64__)
      __builtin_ia32_pause();
#endif
      if (++spins > (1ull << 33)) return false;
    }
  }
  return true;
}
void dist_barrier(DistImpl& D, const char* where) {
  if (!shared_barrier(D.flags, D.rank, D.world, &D.epoch))
    throw StatusError{B2Z_ECUDA, std::string("b2z_dist_prove: a peer rank did not reach the barrier after ") + where};
}
// the last step of a distributed proof: partial sums meet in the shared buffer, every rank combines; the second
// barrier keeps a fast rank from overwriting its slot (next proof) before everybody has read it
bool shared_combine(void* shared_host, uint32_t rank, uint32_t world, uint32_t* epoch, const uint8_t* my_partial,
                    uint8_t proof_out[192]) {
  uint32_t* flags = static_cast<uint32_t*>(shared_host);
  uint8_t* partials = static_cast<uint8_t*>(shared_host) + (size_t)world * kFlagStride * 4;
  if (my_partial != partials + (size_t)rank * kPartial) std::memcpy(partials + (size_t)rank * kPartial, my_partial, kPartial);
  if (!shared_barrier(flags, rank, world, epoch)) return false;
  combine_partials(partials, world, proof_out);
  return shared_barrier(flags, rank, world, epoch);
}
}  // namespace
}  // namespace b2z

struct b2z_dist {
  DistImpl impl;
};

extern "C" {

uint64_t b2z_dist_shared_bytes(uint32_t world) { return (uint64_t)world * (kFlagStride * 4 + kPartial); }

b2z_status b2z_dist_combine_shared(void* shared_host, uint32_t rank, uint32_t world, uint32_t* epoch,
                                   const uint8_t* my_partial, uint8_t proof_out[192]) {
  if (!shared_host || !epoch || !my_partial || !proof_out || world == 0 || rank >= world) return B2Z_EINVAL;
  return shared_combine(shared_host, rank, world, epoch, my_partial, proof_out) ? B2Z_OK : B2Z_ECUDA;
}

b2z_status b2z_dist_create(b2z_ctx* ctx, const b2z_pk* pk, b2z_r1cs* r, uint32_t rank, uint32_t world, void* shared_host,
                           b2z_dist** out) {
  if (out) *out = nullptr;
  return guarded(ctx, [&](Ctx& c) {
    B2Z_REQUIRE(pk && r && shared_host && out, B2Z_EINVAL, "b2z_dist_create: NULL argument");
    B2Z_REQUIRE((world == 2 || world == 4 || world == 8) && rank < world, B2Z_EINVAL,
                "b2z_dist_create: world must be 2, 4 or 8 and rank < world");
    R1csImpl& R = r1cs_of(c, r, "b2z_dist_create");
    PkImpl& P = pk_for(c, pk, R, "b2z_dist_create");
    uint32_t wbits = 0;
    while ((1u << wbits) < world) wbits++;
    B2Z_REQUIRE(ntt_dist_supported(R.log_n, wbits), B2Z_ESIZE,
                "b2z_dist_create: domain too small for a tile-sharded witness map (use b2z_groth16_prove_partial_r1cs)");
    const size_t n = (size_t)1 << R.log_n;
    B2Z_REQUIRE(P.hn == n / world && P.h_lo == n / world * rank, B2Z_EINVAL,
                "b2z_dist_create: the key must be shard `rank` of `world` (b2z_pk_upload_shard)");
    std::unique_ptr<b2z_dist> d(new b2z_dist());
    DistImpl& D = d->impl;
    D.owner = &c; D.rank = rank; D.world = world; D.wbits = wbits; D.log_n = R.log_n; D.m = R.m;
    D.pk = &P; D.r1cs = r;
    D.nl = n / world;
    D.z_bytes = ((R.m * sizeof(FrEl) + 255) / 256) * 256;
    D.region_bytes = D.z_bytes + 6 * D.nl * sizeof(FrEl);
    D.region.alloc(D.region_bytes);
    B2Z_CUDA(cudaMemset(D.region.p, 0, D.region_bytes));
    D.peer_region[rank] = D.region.p;
    D.flags = static_cast<uint32_t*>(shared_host);
    D.partials = static_cast<uint8_t*>(shared_host) + (size_t)world * kFlagStride * 4;
    int lo = 0, hi = 0;
    B2Z_CUDA(cudaDeviceGetStreamPriorityRange(&lo, &hi));
    B2Z_CUDA(cudaStreamCreateWithPriority(&D.wm_st, cudaStreamNonBlocking, hi));
    B2Z_CUDA(cudaEventCreateWithFlags(&D.ev_ready, cudaEventDisableTiming));
    // this rank's rows: local index li of the column-owned layout = global row with the rank inserted at the
    // ownership bits
    {
      const uint32_t ob = ntt_dist_col_bits(R.log_n, wbits);
      auto row_of = [=](uint32_t li) {
        return (uint64_t)(((li >> ob) << (ob + wbits)) | (rank << ob) | (li & ((1u << ob) - 1)));
      };
      for (int k = 0; k < 3; k++) {
        const HostCsr h = download_csr(R.mat[k], R.nc, D.wm_st);
        plan_matrix(D.plan, k, h, R.nc, R.l, (uint32_t)D.nl, row_of, D.wm_st);
      }
      plan_finish(D.plan, (uint32_t)D.nl);
    }
    // warm the twiddle tables now: they are built lazily on first use
    for (TwKind k : {TW_INV, TW_COSET_FWD, TW_COSET_INV}) ntt_twiddles(&c, R.log_n, k, D.wm_st);
    B2Z_CUDA(cudaStreamSynchronize(D.wm_st));
    *out = d.release();
  });
}

void b2z_dist_destroy(b2z_ctx* ctx, b2z_dist* d) {
  if (d == nullptr) return;
  if (ctx != nullptr) {
    std::lock_guard<std::mutex> lock(ctx->impl.mu);
    cudaSetDevice(ctx->impl.device);
    cudaDeviceSynchronize();
  }
  delete d;
}

b2z_status b2z_dist_export(b2z_ctx* ctx, b2z_dist* d, uint8_t ipc_handle[64], void** device_ptr) {
  return guarded(ctx, [&](Ctx& c) {
    B2Z_REQUIRE(d && d->impl.owner == &c && (ipc_handle || device_ptr), B2Z_EINVAL, "b2z_dist_export: bad argument");
    if (device_ptr) *device_ptr = d->impl.region.p;
    if (ipc_handle) {
      cudaIpcMemHandle_t h;
      static_assert(sizeof(h) == 64, "cudaIpcMemHandle_t is 64 bytes");
      B2Z_CUDA(cudaIpcGetMemHandle(&h, d->impl.region.p));
      std::memcpy(ipc_handle, &h, 64);
    }
  });
}

b2z_status b2z_dist_attach(b2z_ctx* ctx, b2z_dist* d, uint32_t peer, const uint8_t* ipc_handle, void* device_ptr) {
  return guarded(ctx, [&](Ctx& c) {
    B2Z_REQUIRE(d && d->impl.owner == &c && peer < d->impl.world && (ipc_handle != nullptr) != (device_ptr != nullptr),
                B2Z_EINVAL, "b2z_dist_attach: need a peer rank and exactly one of ipc_handle / device_ptr");
    DistImpl& D = d->impl;
    if (peer == D.rank) return;
    if (device_ptr != nullptr) {
      // same process: a plain device pointer; enable peer access when it lives on another GPU
      cudaPointerAttributes at;
      B2Z_CUDA(cudaPointerGetAttributes(&at, device_ptr));
      if (at.device != c.device) {
        const cudaError_t e = cudaDeviceEnablePeerAccess(at.device, 0);
        if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) B2Z_CUDA(e);
        cudaGetLastError();
      }
      D.peer_region[peer] = static_cast<uint8_t*>(device_ptr);
    } else {
      cudaIpcMemHandle_t h;
      std::memcpy(&h, ipc_handle, 64);
      void* p = nullptr;
      B2Z_CUDA(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
      D.peer_region[peer] = static_cast<uint8_t*>(p);
      D.peer_ipc[peer] = true;
    }
  });
}

b2z_status b2z_dist_prove(b2z_ctx* ctx, b2z_dist* d, const uint64_t* z, int z_is_full_device_copy, const uint64_t rr[4],
                          const uint64_t ss[4], uint8_t proof_out[192]) {
  return guarded(ctx, [&](Ctx& c) {
    B2Z_REQUIRE(d && d->impl.owner == &c && z && rr && ss && proof_out, B2Z_EINVAL, "b2z_dist_prove: bad argument");
    DistImpl& D = d->impl;
    for (uint32_t p = 0; p < D.world; p++)
      B2Z_REQUIRE(D.peer_region[p] != nullptr, B2Z_EINVAL, "b2z_dist_prove: not every peer is attached (b2z_dist_attach)");
    R1csImpl& R = r1cs_of(c, D.r1cs, "b2z_dist_prove");
    PkImpl& P = *D.pk;
    cudaStream_t ws = D.wm_st;
    // ---- the assignment: every rank moves 1 / W of it over PCIe and hands the slice to its peers over NVLink
    if (z_is_full_device_copy) {
      B2Z_CUDA(cudaMemcpyAsync(D.z(), z, D.m * sizeof(FrEl), cudaMemcpyDefault, ws));
    } else {
      const uint64_t lo = D.m * D.rank / D.world, hi = D.m * (D.rank + 1) / D.world;
      const size_t off = lo * sizeof(FrEl), bytes = (hi - lo) * sizeof(FrEl);
      B2Z_CUDA(cudaMemcpyAsync(D.region.p + off, reinterpret_cast<const uint8_t*>(z) + off, bytes, cudaMemcpyDefault, ws));
      if (bytes) {
        PeerPtrs pp;
        for (uint32_t k = 1; k < D.world; k++)
          pp.p[k - 1] = reinterpret_cast<uint4*>(D.peer_region[(D.rank + k) % D.world] + off);
        z_scatter_kernel<<<296, 256, 0, ws>>>(reinterpret_cast<const uint4*>(D.region.p + off), bytes / 16, pp, D.world - 1);
        B2Z_LAUNCHED(&c);
      }
      B2Z_CUDA(cudaStreamSynchronize(ws));
      dist_barrier(D, "the assignment exchange");
    }
    B2Z_CUDA(cudaEventRecord(R.ev_z, ws));
    // ---- light z-only work on the auxiliary streams: scalar conversion and the four sorts
    B2Z_CUDA(cudaStreamWaitEvent(c.aux[0], R.ev_z, 0));
    proof_begin(c, P, D.z(), rr, ss);
    // ---- tile-sharded witness map on its own high-priority stream
    NttDist& nd = D.nd;
    nd.wbits = D.wbits; nd.me = D.rank;
    for (int v = 0; v < 3; v++) {
      nd.x[v] = reinterpret_cast<FrEl*>(D.vec_of(D.region.p, 0, v));
      nd.y[v] = reinterpret_cast<FrEl*>(D.vec_of(D.region.p, 1, v));
      for (uint32_t p = 0; p < D.world; p++) {
        nd.peer_x[v][p] = reinterpret_cast<FrEl*>(D.vec_of(D.peer_region[p], 0, v));
        nd.peer_y[v][p] = reinterpret_cast<FrEl*>(D.vec_of(D.peer_region[p], 1, v));
      }
    }
    run_plan(c, D.plan, D.z(), nd.x[0], nd.x[1], nd.x[2], ws);
    wm_dist_step1(&c, nd, D.log_n, ws);
    B2Z_CUDA(cudaStreamSynchronize(ws));
    dist_barrier(D, "witness-map step 1");
    wm_dist_step2(&c, nd, D.log_n, ws);
    B2Z_CUDA(cudaStreamSynchronize(ws));
    dist_barrier(D, "witness-map step 2");
    wm_dist_step3(&c, nd, D.log_n, ws);
    B2Z_CUDA(cudaStreamSynchronize(ws));
    dist_barrier(D, "witness-map step 3");
    wm_dist_step4(&c, nd, D.log_n, ws);
    B2Z_CUDA(cudaEventRecord(D.ev_ready, ws));
    proof_h_sort(c, P, nd.y[0], ws);                       // hides under the z-only accumulations
    // ---- the five accumulations back to back once the transforms are done (they need the SMs the accumulations
    // fill), H on ws after its sort; host epilogue of this shard
    proof_accums(c, P, D.ev_ready);
    proof_h_finish(c, P);
    proof_end(c, P, D.partials + (size_t)D.rank * kPartial);
    // ---- partial sums meet in the shared host memory; every rank combines
    if (!shared_combine(D.flags, D.rank, D.world, &D.epoch, D.partials + (size_t)D.rank * kPartial, proof_out))
      throw StatusError{B2Z_ECUDA, "b2z_dist_prove: a peer rank did not reach the barrier after the accumulations"};
  });
}

}  // extern "C"
