// pc_solve.cu -- the step AFTER the assembly path (SURVEY 8 f-4): a device-resident consumer of the assembled CSR, so that a
// caller can assemble and solve without one matrix byte crossing PCIe.
//
// In the reference the assembled Mat goes to PETSc: IGACreateKSP (src/petiga.c:856-885) + KSPSetOperators + KSPSolve
// (demo/Poisson3D.c:73-83, run with -ksp_type cg -pc_type jacobi in demo/makefile's Poisson targets).  PETSc is not part of this
// build, so the same two pieces are provided on the device for the matrix layouts the path writes:
//   petiga_cuda_spmv      y = A x          (MatMult)   AIJ scalar CSR or BAIJ block CSR with column-major blocks
//   petiga_cuda_solve_cg  Jacobi-preconditioned conjugate gradients (KSPCG + PCJACOBI), scalars kept on the device:
//                         one host read of the residual norm every `check` iterations, none otherwise
//   petiga_cuda_solve_gmres  restarted GMRES with the Jacobi diagonal on the right (KSPGMRES + PCJACOBI, -ksp_pc_side right) for
//                         the non-symmetric Jacobians; the same host-read cadence, convergence decided on the true residual
// Multi-rank: rows are distributed as the matrix is (rank-major global numbering, src/petigagrid.c:98-171); the operand of
// the product is gathered into a full-length device vector over NCCL (a grouped ncclBroadcast per owner: the VecScatter of
// MatMult_MPIAIJ), dot products by ncclAllReduce.  Deterministic: every reduction is a fixed-shape tree.
#include <cmath>
#include <cstring>
#include <vector>

#include "pc_plan.h"

namespace pc {

namespace {

constexpr int kDotBlocks = 512;

// one warp per scalar row (AIJ) -- 12 bytes of matrix per nonzero, the x gathers hit L2 (x is 18 MB at cfg 2); measured at cfg 2
// (tools/solve_probe.py): 1.79 -> 1.64 ms per CG iteration with evict-first loads of the matrix
__global__ void __launch_bounds__(256) spmv_aij_kernel(int nrows, const int* __restrict__ rowptr, const int* __restrict__ colidx,
                                                       const double* __restrict__ values, const double* __restrict__ x, double* __restrict__ y) {
  const int lane = threadIdx.x & 31, wpb = blockDim.x >> 5;
  for (int row = blockIdx.x * wpb + (threadIdx.x >> 5); row < nrows; row += gridDim.x * wpb) {
    const int s = rowptr[row], e = rowptr[row + 1];
    double acc = 0.0;
    // the matrix streams through once per product: evict-first loads keep the operand vector (18 MB at cfg 2) resident in L2
    for (int k = s + lane; k < e; k += 32) acc = fma(__ldcs(values + k), __ldg(x + __ldcs(colidx + k)), acc);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) y[row] = acc;
  }
}

// one warp per block row (BAIJ, bs x bs column-major blocks): lane t walks the scalars of the row's blocks
template <int BS>
__global__ void __launch_bounds__(256) spmv_baij_kernel(int nrows, const int* __restrict__ rowptr, const int* __restrict__ colidx,
                                                        const double* __restrict__ values, const double* __restrict__ x, double* __restrict__ y) {
  const int lane = threadIdx.x & 31, wpb = blockDim.x >> 5;
  for (int row = blockIdx.x * wpb + (threadIdx.x >> 5); row < nrows; row += gridDim.x * wpb) {
    const int64_t s = (int64_t)rowptr[row] * BS * BS, e = (int64_t)rowptr[row + 1] * BS * BS;
    double acc[BS];
#pragma unroll
    for (int i = 0; i < BS; i++) acc[i] = 0.0;
    for (int64_t k = s + lane; k < e; k += 32) {
      const int64_t blk = k / (BS * BS);
      const int r = (int)(k - blk * BS * BS), i = r % BS, j = r / BS;
      const double v = __ldcs(values + k) * __ldg(x + (size_t)__ldcs(colidx + blk) * BS + j);
#pragma unroll
      for (int ii = 0; ii < BS; ii++) if (ii == i) acc[ii] += v;
    }
#pragma unroll
    for (int i = 0; i < BS; i++) {
      double a = acc[i];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
      if (lane == 0) y[(size_t)row * BS + i] = a;
    }
  }
}

// 1 / diagonal (PCJACOBI); `grow0` = first global scalar row of this rank
__global__ void diag_inv_kernel(int nrows, int bs, int grow0, const int* __restrict__ rowptr, const int* __restrict__ colidx,
                                const double* __restrict__ values, double* __restrict__ dinv) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;          // scalar row
  if (r >= nrows * bs) return;
  double d = 0.0;
  if (bs == 1) {
    const int g = grow0 + r;
    for (int k = rowptr[r]; k < rowptr[r + 1]; k++) if (colidx[k] == g) d = values[k];
  } else {
    const int br = r / bs, i = r - br * bs, g = grow0 / bs + br;
    for (int k = rowptr[br]; k < rowptr[br + 1]; k++) if (colidx[k] == g) d = values[(size_t)k * bs * bs + i * bs + i];
  }
  dinv[r] = d != 0.0 ? 1.0 / d : 1.0;
}

// fixed-shape dot products: partial[b] per block (tree inside the block), then one block folds the partials in index order
template <int NV>
__device__ __forceinline__ void block_fold(double (&v)[NV], double* part, int nparts_stride) {
  __shared__ double sh[NV][8];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int q = 0; q < NV; q++) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v[q] += __shfl_xor_sync(0xffffffffu, v[q], o);
    if (lane == 0) sh[q][warp] = v[q];
  }
  __syncthreads();
  if (threadIdx.x < NV) {
    double a = 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); w++) a += sh[threadIdx.x][w];
    part[threadIdx.x * nparts_stride + blockIdx.x] = a;
  }
}
// one block folds every quantity (CG), or one block per quantity (GMRES's batch of dot products); either way each sum has the
// same fixed order
__global__ void __launch_bounds__(256) fold_partials_kernel(const double* __restrict__ part, int nparts, int nv, double* __restrict__ out) {
  __shared__ double sh[256];
  for (int q = blockIdx.x; q < nv; q += gridDim.x) {
    double a = 0.0;
    for (int i = threadIdx.x; i < nparts; i += 256) a += part[q * nparts + i];
    sh[threadIdx.x] = a;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) { if ((int)threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o]; __syncthreads(); }
    if (threadIdx.x == 0) out[q] = sh[0];
    __syncthreads();
  }
}
// out[0] = a.b, out[1] = c.d (two dot products in one pass)
__global__ void __launch_bounds__(256) dot2_kernel(int n, const double* __restrict__ a, const double* __restrict__ b, const double* __restrict__ c,
                                                   const double* __restrict__ d, double* __restrict__ part) {
  double v[2] = {0.0, 0.0};
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) { v[0] = fma(a[i], b[i], v[0]); v[1] = fma(c[i], d[i], v[1]); }
  block_fold<2>(v, part, gridDim.x);
}
// s = [rho, pAp, ...]: x += alpha p, r -= alpha Ap, z = dinv r;  partials of (r.z, r.r);  alpha = s[0] / s[1]
__global__ void __launch_bounds__(256) cg_update_kernel(int n, const double* __restrict__ s, const double* __restrict__ p, const double* __restrict__ Ap,
                                                        const double* __restrict__ dinv, double* __restrict__ x, double* __restrict__ r,
                                                        double* __restrict__ z, double* __restrict__ part) {
  const double alpha = s[0] / s[1];
  double v[2] = {0.0, 0.0};
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    x[i] = fma(alpha, p[i], x[i]);
    const double ri = fma(-alpha, Ap[i], r[i]);
    const double zi = dinv[i] * ri;
    r[i] = ri; z[i] = zi;
    v[0] = fma(ri, zi, v[0]); v[1] = fma(ri, ri, v[1]);
  }
  block_fold<2>(v, part, gridDim.x);
}
// p = z + (rho_new / rho) p ; then rho <- rho_new.  s[0] = rho, s[2] = rho_new
__global__ void __launch_bounds__(256) cg_direction_kernel(int n, const double* __restrict__ s, const double* __restrict__ z, double* __restrict__ p) {
  const double beta = s[2] / s[0];
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) p[i] = fma(beta, p[i], z[i]);
}
__global__ void cg_shift_kernel(double* s) { s[0] = s[2]; }
__global__ void axpby_kernel(int n, double a, const double* __restrict__ x, double b, double* __restrict__ y) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) y[i] = a * x[i] + b * y[i];
}
__global__ void mul_kernel(int n, const double* __restrict__ a, const double* __restrict__ b, double* __restrict__ y) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) y[i] = a[i] * b[i];
}

// ---- GMRES(m) with right Jacobi preconditioning ----
// Scalars of a solve, kept on the device next to the Hessenberg matrix so that the host reads them with one copy.
enum GmresState { kScale = 0, kEst, kFlag, kValid, kExec, kBeta2, kBnorm2, kWnorm2, kStateLen };
// kFlag: why the Arnoldi burst stopped early (later kernels of the burst see it and return at once)
enum GmresStop { kRunning = 0, kEstimateMet = 1, kHappy = 2, kSingular = 3, kNonFinite = 4 };

// v_k = scale w (k >= 1; v_0 = r / beta), z = D^-1 v_k
__global__ void __launch_bounds__(256) gmres_basis_kernel(int n, const double* __restrict__ st, const double* __restrict__ w,
                                                          const double* __restrict__ dinv, double* __restrict__ vk, double* __restrict__ z) {
  if (st[kFlag] != kRunning) return;
  const double scale = st[kScale];
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const double v = w[i] * scale;
    vk[i] = v; z[i] = dinv[i] * v;
  }
}
// h_j = v_{j0+j} . w for j < nv <= KC: one pass over the basis, w read once per row, partials [KC][blocks]
template <int KC>
__global__ void __launch_bounds__(256) gmres_dot_kernel(int n, int nv, const double* __restrict__ st, const double* __restrict__ V, size_t ld,
                                                        const double* __restrict__ w, double* __restrict__ part) {
  if (st[kFlag] != kRunning) return;
  double acc[KC];
#pragma unroll
  for (int j = 0; j < KC; j++) acc[j] = 0.0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const double wi = w[i];
#pragma unroll
    for (int j = 0; j < KC; j++) if (j < nv) acc[j] = fma(V[j * ld + i], wi, acc[j]);
  }
  block_fold<KC>(acc, part, gridDim.x);
}
// w -= sum_j h_j v_j (j <= k, classical Gram-Schmidt) and the partials of |w|^2
__global__ void __launch_bounds__(256) gmres_update_kernel(int n, int nv, const double* __restrict__ st, const double* __restrict__ V, size_t ld,
                                                           const double* __restrict__ h, double* __restrict__ w, double* __restrict__ part) {
  if (st[kFlag] != kRunning) return;
  double v[1] = {0.0};
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    double s = 0.0;
    for (int j = 0; j < nv; j++) s = fma(h[j], V[j * ld + i], s);
    const double wi = w[i] - s;
    w[i] = wi;
    v[0] = fma(wi, wi, v[0]);
  }
  block_fold<1>(v, part, gridDim.x);
}
// start of a cycle: g = beta e_1, v_0 = r / beta
__global__ void gmres_start_kernel(int m, double* __restrict__ st, double* __restrict__ g) {
  if (threadIdx.x != 0) return;
  const double beta = sqrt(st[kBeta2]);
  for (int i = 0; i <= m; i++) g[i] = 0.0;
  g[0] = beta;
  st[kScale] = 1.0 / beta; st[kEst] = beta;
  st[kFlag] = kRunning; st[kValid] = 0; st[kExec] = 0;
}
// Arnoldi tail of column k (one warp; the work is O(k)): store the column of H, apply the earlier Givens rotations, make the new one,
// update g and the residual estimate |g_{k+1}|, and raise the stop flag.  Nothing non-finite is stored: such a column stops the
// burst with kNonFinite before it counts, so the solution update only ever sees finite columns.
__global__ void gmres_tail_kernel(int k, int m, double target, const double* __restrict__ hd, double* __restrict__ st, double* __restrict__ H,
                                  double* __restrict__ cs, double* __restrict__ sn, double* __restrict__ g) {
  if (threadIdx.x != 0 || st[kFlag] != kRunning) return;
  st[kExec] = k + 1;
  const double hn = sqrt(st[kWnorm2]);
  bool finite = isfinite(hn);
  for (int i = 0; i <= k; i++) finite = finite && isfinite(hd[i]);
  if (!finite) { st[kFlag] = kNonFinite; return; }
  double* col = H + (size_t)k * (m + 1);
  for (int i = 0; i <= k; i++) col[i] = hd[i];
  col[k + 1] = hn;
  for (int i = 0; i < k; i++) {
    const double a = col[i], b = col[i + 1];
    col[i] = cs[i] * a + sn[i] * b;
    col[i + 1] = -sn[i] * a + cs[i] * b;
  }
  const double r = hypot(col[k], hn);
  if (!(r > 0.0)) { st[kFlag] = kSingular; return; }          // A D^-1 v_k = 0: the column cannot enter the least-squares solve
  cs[k] = col[k] / r; sn[k] = hn / r;
  col[k] = r; col[k + 1] = 0.0;
  g[k + 1] = -sn[k] * g[k];
  g[k] = cs[k] * g[k];
  st[kValid] = k + 1;
  st[kEst] = fabs(g[k + 1]);
  st[kScale] = hn > 0.0 ? 1.0 / hn : 0.0;
  if (hn == 0.0) st[kFlag] = kHappy;
  else if (fabs(g[k + 1]) <= target) st[kFlag] = kEstimateMet;
}
// y = R^-1 g over the first kv columns (back substitution, one thread)
__global__ void gmres_ysolve_kernel(int kv, int m, const double* __restrict__ H, const double* __restrict__ g, double* __restrict__ y) {
  if (threadIdx.x != 0) return;
  for (int i = kv - 1; i >= 0; i--) {
    double s = g[i];
    for (int j = i + 1; j < kv; j++) s -= H[(size_t)j * (m + 1) + i] * y[j];
    y[i] = s / H[(size_t)i * (m + 1) + i];
  }
}
// x += D^-1 V y
__global__ void __launch_bounds__(256) gmres_xupdate_kernel(int n, int kv, const double* __restrict__ V, size_t ld, const double* __restrict__ y,
                                                            const double* __restrict__ dinv, double* __restrict__ x) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    double s = 0.0;
    for (int j = 0; j < kv; j++) s = fma(y[j], V[j * ld + i], s);
    x[i] = fma(dinv[i], s, x[i]);
  }
}

struct Pattern { int nrows; int64_t nnz; const int* rowptr; const int* colidx; int bs; };

int get_pattern(petiga_cuda_plan* P, int block, Pattern& pt) {
  int rc = petiga_cuda_plan_pattern(P, block, &pt.nrows, &pt.nnz, &pt.rowptr, &pt.colidx);
  pt.bs = block ? P->L.dof : 1;
  return rc;
}

// operand of the product: the owned slice on one rank, else gathered into the plan's full-length buffer
int full_operand(petiga_cuda_plan* P, const double* x_owned, const double** xfull) {
  const Layout& L = P->L;
  if (L.nranks == 1) { *xfull = x_owned; return 0; }
  const size_t ntot = (size_t)L.rank_start[L.nranks] * L.dof;
  int rc = P->d_solve_xfull.reserve(ntot);
  if (rc) return rc;
  rc = allgather_owned(P, x_owned, P->d_solve_xfull.get());
  if (rc) return rc;
  *xfull = P->d_solve_xfull.get();
  return 0;
}

int spmv(petiga_cuda_plan* P, const Pattern& pt, const double* values, const double* x_owned, double* y) {
  const double* xf = nullptr;
  int rc = full_operand(P, x_owned, &xf);
  if (rc) return rc;
  if (pt.nrows <= 0) return 0;
  const int blocks = std::max(1, std::min((pt.nrows + 7) / 8, P->num_sms * 16));
  if (pt.bs == 1) spmv_aij_kernel<<<blocks, 256, 0, P->stream>>>(pt.nrows, pt.rowptr, pt.colidx, values, xf, y);
  else if (pt.bs == 2) spmv_baij_kernel<2><<<blocks, 256, 0, P->stream>>>(pt.nrows, pt.rowptr, pt.colidx, values, xf, y);
  else if (pt.bs == 3) spmv_baij_kernel<3><<<blocks, 256, 0, P->stream>>>(pt.nrows, pt.rowptr, pt.colidx, values, xf, y);
  else if (pt.bs == 4) spmv_baij_kernel<4><<<blocks, 256, 0, P->stream>>>(pt.nrows, pt.rowptr, pt.colidx, values, xf, y);
  else { set_error("spmv: block size > 4 (use the AIJ layout)"); return PETIGA_CUDA_ERR_SUP; }
  PC_CUDA(cudaGetLastError());
  P->launches++;
  return 0;
}

}  // namespace

}  // namespace pc

using namespace pc;

extern "C" int petiga_cuda_spmv(petiga_cuda_plan* P, int block, const double* values, const double* x, double* y) {
  if (!P || !values || !x || !y) return PETIGA_CUDA_ERR_ARG;
  PC_CUDA(cudaSetDevice(P->device));
  nvtx_push("petiga_cuda_spmv");
  struct Pop { ~Pop() { nvtx_pop(); } } pop;
  Pattern pt;
  int rc = get_pattern(P, block, pt);
  if (rc) return rc;
  return spmv(P, pt, values, x, y);          // enqueued on the plan's stream; petiga_cuda_finish waits
}

extern "C" int petiga_cuda_solve_cg(petiga_cuda_plan* P, int block, const double* values, const double* b, double* x, double rtol, double atol,
                                    int maxit, int* iters_out, double* relres_out) {
  if (!P || !values || !b || !x || maxit < 0) return PETIGA_CUDA_ERR_ARG;
  PC_CUDA(cudaSetDevice(P->device));
  nvtx_push("petiga_cuda_solve_cg");
  struct Pop { ~Pop() { nvtx_pop(); } } pop;
  const Layout& L = P->L;
  Pattern pt;
  int rc = get_pattern(P, block, pt);
  if (rc) return rc;
  const int n = pt.nrows * pt.bs;                       // owned scalar rows
  // work vectors r, z, p, Ap, dinv + partials + scalars, kept with the plan
  const size_t need = (size_t)5 * std::max(n, 1) + 4 * kDotBlocks + 16;
  if ((rc = P->d_solve_work.reserve(need))) return rc;
  double *r = P->d_solve_work.get(), *z = r + n, *p = z + n, *Ap = p + n, *dinv = Ap + n, *part = dinv + n, *s = part + 4 * kDotBlocks;
  cudaStream_t st = P->stream;
  const int gb = std::max(1, std::min((n + 255) / 256, kDotBlocks));
  const bool multi = L.nranks > 1;
  auto reduce = [&](int nv, double* out) -> int {      // partials -> out[0..nv) (+ sum over ranks)
    fold_partials_kernel<<<1, 256, 0, st>>>(part, gb, nv, out);
    PC_CUDA(cudaGetLastError());
    if (multi) return allreduce_sum(P, out, nv);
    return 0;
  };
  if (n > 0) diag_inv_kernel<<<(n + 255) / 256, 256, 0, st>>>(pt.nrows, pt.bs, L.rank_start[L.rank] * L.dof, pt.rowptr, pt.colidx, values, dinv);
  // r = b - A x
  if ((rc = spmv(P, pt, values, x, Ap))) return rc;
  PC_CUDA(cudaMemcpyAsync(r, b, (size_t)n * sizeof(double), cudaMemcpyDeviceToDevice, st));
  axpby_kernel<<<gb, 256, 0, st>>>(n, -1.0, Ap, 1.0, r);
  mul_kernel<<<gb, 256, 0, st>>>(n, dinv, r, z);
  PC_CUDA(cudaMemcpyAsync(p, z, (size_t)n * sizeof(double), cudaMemcpyDeviceToDevice, st));
  dot2_kernel<<<gb, 256, 0, st>>>(n, r, z, b, b, part);            // rho = r.z, |b|^2
  if ((rc = reduce(2, s + 4))) return rc;                           // s[4] = rho, s[5] = |b|^2
  dot2_kernel<<<gb, 256, 0, st>>>(n, r, r, r, r, part);
  if ((rc = reduce(1, s + 6))) return rc;                           // s[6] = |r0|^2
  double h[3];
  PC_CUDA(cudaMemcpyAsync(h, s + 4, 3 * sizeof(double), cudaMemcpyDeviceToHost, st));
  PC_CUDA(cudaStreamSynchronize(st));
  const double bnorm = std::sqrt(h[1]);
  double rnorm = std::sqrt(h[2]);
  const double target = std::max(rtol * (bnorm > 0 ? bnorm : 1.0), atol);
  PC_CUDA(cudaMemcpyAsync(s, s + 4, sizeof(double), cudaMemcpyDeviceToDevice, st));    // s[0] = rho
  int it = 0;
  const int check = 10;
  while (it < maxit && rnorm > target) {
    const int burst = std::min(check, maxit - it);
    for (int k = 0; k < burst; k++) {
      if ((rc = spmv(P, pt, values, p, Ap))) return rc;
      dot2_kernel<<<gb, 256, 0, st>>>(n, p, Ap, p, Ap, part);
      if ((rc = reduce(1, s + 1))) return rc;                                           // s[1] = p.Ap
      cg_update_kernel<<<gb, 256, 0, st>>>(n, s, p, Ap, dinv, x, r, z, part);
      if ((rc = reduce(2, s + 2))) return rc;                                           // s[2] = rho_new, s[3] = |r|^2
      cg_direction_kernel<<<gb, 256, 0, st>>>(n, s, z, p);
      cg_shift_kernel<<<1, 1, 0, st>>>(s);
      P->launches += 6;
    }
    it += burst;
    PC_CUDA(cudaMemcpyAsync(h, s + 3, sizeof(double), cudaMemcpyDeviceToHost, st));
    PC_CUDA(cudaStreamSynchronize(st));
    rnorm = std::sqrt(h[0]);
    if (!(rnorm == rnorm)) { set_error("solve_cg: breakdown (the matrix is not symmetric positive definite?)"); return PETIGA_CUDA_ERR_ARG; }
  }
  PC_CUDA(cudaGetLastError());
  if (iters_out) *iters_out = it;
  if (relres_out) *relres_out = bnorm > 0 ? rnorm / bnorm : rnorm;
  return 0;
}

extern "C" int petiga_cuda_solve_gmres(petiga_cuda_plan* P, int block, const double* values, const double* b, double* x, int restart, double rtol,
                                       double atol, int maxit, int* iters_out, double* relres_out, int* reason_out) {
  if (!P || !values || !b || !x || !iters_out || !relres_out || !reason_out || b == x || restart < 1 || maxit < 0) return PETIGA_CUDA_ERR_ARG;
  PC_CUDA(cudaSetDevice(P->device));
  nvtx_push("petiga_cuda_solve_gmres");
  struct Pop { ~Pop() { nvtx_pop(); } } pop;
  const Layout& L = P->L;
  Pattern pt;
  int rc = get_pattern(P, block, pt);
  if (rc) return rc;
  if (pt.bs > 4) { set_error("solve_gmres: block size > 4 (use the AIJ layout)"); return PETIGA_CUDA_ERR_SUP; }
  const int n = pt.nrows * pt.bs, m = restart;
  const size_t ld = (size_t)std::max(n, 1);
  const int kc = 32;                                           // basis vectors per pass of the multi-dot
  const int npass = (m + 1 + kc - 1) / kc;
  // basis V[m+1], w, z, 1/diag, partials [npass*32][blocks], H[m][m+1], cs, sn, g, y, h, state; kept with the plan
  const size_t nsmall = (size_t)m * (m + 1) + 2 * (size_t)m + 2 * (size_t)(m + 1) + (size_t)npass * kc + kStateLen;
  const size_t need = (size_t)(m + 4) * ld + (size_t)npass * kc * kDotBlocks + nsmall;
  if ((rc = P->d_gmres_work.reserve(need))) return rc;
  double *V = P->d_gmres_work.get(), *w = V + (size_t)(m + 1) * ld, *z = w + ld, *dinv = z + ld, *part = dinv + ld;
  double *H = part + (size_t)npass * kc * kDotBlocks, *cs = H + (size_t)m * (m + 1), *sn = cs + m, *g = sn + m, *y = g + m + 1;
  double *hd = y + m + 1, *st = hd + (size_t)npass * kc;
  cudaStream_t s = P->stream;
  const int gb = std::max(1, std::min((n + 255) / 256, kDotBlocks));
  const bool multi = L.nranks > 1;
  auto reduce = [&](int nv, double* out) -> int {              // partials -> out[0..nv) (+ sum over ranks)
    fold_partials_kernel<<<nv, 256, 0, s>>>(part, gb, nv, out);
    PC_CUDA(cudaGetLastError());
    P->launches++;
    return multi ? allreduce_sum(P, out, nv) : 0;
  };
  auto true_residual = [&]() -> int {                          // w = b - A x, st[kBeta2] = |w|^2
    if (int e = spmv(P, pt, values, x, w)) return e;
    axpby_kernel<<<gb, 256, 0, s>>>(n, 1.0, b, -1.0, w);
    dot2_kernel<<<gb, 256, 0, s>>>(n, w, w, w, w, part);
    P->launches += 2;
    return reduce(1, st + kBeta2);
  };
  double h[kStateLen];
  auto read_state = [&]() -> int {
    PC_CUDA(cudaMemcpyAsync(h, st, sizeof(h), cudaMemcpyDeviceToHost, s));
    PC_CUDA(cudaStreamSynchronize(s));
    return 0;
  };

  if (n > 0) diag_inv_kernel<<<(n + 255) / 256, 256, 0, s>>>(pt.nrows, pt.bs, L.rank_start[L.rank] * L.dof, pt.rowptr, pt.colidx, values, dinv);
  dot2_kernel<<<gb, 256, 0, s>>>(n, b, b, b, b, part);
  P->launches += 2;
  if ((rc = reduce(1, st + kBnorm2))) return rc;
  if ((rc = true_residual()) || (rc = read_state())) return rc;
  const double bnorm = std::sqrt(h[kBnorm2]);
  const double target = std::max(rtol * bnorm, atol);
  *iters_out = 0; *relres_out = 0.0;
  if (!std::isfinite(bnorm)) { *relres_out = bnorm; *reason_out = PETIGA_KSP_DIVERGED_NANORINF; return 0; }
  if (bnorm == 0.0) {                                          // b = 0: the solution is x = 0 (KSPSolve does the same)
    PC_CUDA(cudaMemsetAsync(x, 0, (size_t)n * sizeof(double), s));
    PC_CUDA(cudaStreamSynchronize(s));
    *reason_out = PETIGA_KSP_CONVERGED_ATOL;
    return 0;
  }
  int its = 0, stop = kRunning;
  const int check = 10;
  for (;;) {
    // convergence is decided on the true residual only, once per cycle
    const double rnorm = std::sqrt(h[kBeta2]);
    *relres_out = rnorm / bnorm;
    if (!std::isfinite(rnorm)) { *reason_out = PETIGA_KSP_DIVERGED_NANORINF; break; }
    if (rnorm <= target) { *reason_out = rnorm <= rtol * bnorm ? PETIGA_KSP_CONVERGED_RTOL : PETIGA_KSP_CONVERGED_ATOL; break; }
    if (stop == kNonFinite) { *reason_out = PETIGA_KSP_DIVERGED_NANORINF; break; }
    if (stop == kHappy || stop == kSingular) { *reason_out = PETIGA_KSP_DIVERGED_BREAKDOWN; break; }
    if (its >= maxit) { *reason_out = PETIGA_KSP_DIVERGED_ITS; break; }
    gmres_start_kernel<<<1, 32, 0, s>>>(m, st, g);
    P->launches++;
    int k = 0;
    stop = kRunning;
    while (stop == kRunning && k < m && its + k < maxit) {
      const int burst = std::min(check, std::min(m - k, maxit - its - k));
      for (int q = k; q < k + burst; q++) {
        gmres_basis_kernel<<<gb, 256, 0, s>>>(n, st, w, dinv, V + q * ld, z);
        if ((rc = spmv(P, pt, values, z, w))) return rc;
        for (int p = 0; p * kc <= q; p++) {
          const int nv = std::min(kc, q + 1 - p * kc);
          const double* Vp = V + (size_t)p * kc * ld;
          double* pp = part + (size_t)p * kc * gb;
          if (nv <= 8) gmres_dot_kernel<8><<<gb, 256, 0, s>>>(n, nv, st, Vp, ld, w, pp);
          else if (nv <= 16) gmres_dot_kernel<16><<<gb, 256, 0, s>>>(n, nv, st, Vp, ld, w, pp);
          else gmres_dot_kernel<32><<<gb, 256, 0, s>>>(n, nv, st, Vp, ld, w, pp);
          P->launches++;
        }
        if ((rc = reduce(q + 1, hd))) return rc;
        gmres_update_kernel<<<gb, 256, 0, s>>>(n, q + 1, st, V, ld, hd, w, part);
        if ((rc = reduce(1, st + kWnorm2))) return rc;
        gmres_tail_kernel<<<1, 32, 0, s>>>(q, m, target, hd, st, H, cs, sn, g);
        P->launches += 3;
      }
      if ((rc = read_state())) return rc;
      stop = (int)h[kFlag];
      k = (int)h[kExec];
    }
    its += k;
    const int kv = (int)h[kValid];
    if (kv > 0) {
      gmres_ysolve_kernel<<<1, 32, 0, s>>>(kv, m, H, g, y);
      gmres_xupdate_kernel<<<gb, 256, 0, s>>>(n, kv, V, ld, y, dinv, x);
      P->launches += 2;
    }
    if ((rc = true_residual()) || (rc = read_state())) return rc;
  }
  PC_CUDA(cudaGetLastError());
  *iters_out = its;
  return 0;
}
