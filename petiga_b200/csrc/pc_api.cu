// pc_api.cu -- extern "C" entry points of libpetiga_cuda (see include/petiga_cuda.h).
#include <dlfcn.h>

#include <sched.h>

#include <algorithm>
#include <cctype>
#include <cstdio>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "pc_plan.h"

namespace pc {

// NVTX ranges around the driver bodies (SURVEY 5: tracing).  libnvToolsExt is loaded lazily with dlopen so that the library has
// no link-time dependency on it; without it the ranges are no-ops.
namespace {
typedef int (*nvtx_push_t)(const char*);
typedef int (*nvtx_pop_t)(void);
nvtx_push_t g_nvtx_push = nullptr;
nvtx_pop_t g_nvtx_pop = nullptr;
int g_nvtx_state = 0;   // 0 untried, 1 loaded, -1 unavailable
const char* const kSlotNames[PETIGA_NSLOTS] = {"IGAComputeVector", "IGAComputeMatrix", "IGAComputeSystem", "IGAComputeFunction", "IGAComputeJacobian",
                                               "IGAComputeIFunction", "IGAComputeIJacobian", "IGAComputeIEFunction", "IGAComputeIEJacobian",
                                               "IGAComputeRHSFunction", "IGAComputeRHSJacobian", "IGAComputeI2Function", "IGAComputeI2Jacobian"};
void nvtx_init() {
  if (g_nvtx_state) return;
  g_nvtx_state = -1;
  for (const char* n : {"libnvToolsExt.so.1", "libnvToolsExt.so"}) {
    void* h = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
    if (!h) continue;
    g_nvtx_push = (nvtx_push_t)dlsym(h, "nvtxRangePushA");
    g_nvtx_pop = (nvtx_pop_t)dlsym(h, "nvtxRangePop");
    if (g_nvtx_push && g_nvtx_pop) { g_nvtx_state = 1; return; }
  }
}
}  // namespace
void nvtx_push(int slot) { nvtx_init(); if (g_nvtx_state == 1) g_nvtx_push(kSlotNames[slot]); }
void nvtx_push(const char* name) { nvtx_init(); if (g_nvtx_state == 1) g_nvtx_push(name); }
void nvtx_pop() { if (g_nvtx_state == 1) g_nvtx_pop(); }

static thread_local std::string g_last_error;
void set_error(const std::string& msg) { g_last_error = msg; }
int cuda_fail(cudaError_t e, const char* what) {
  g_last_error = std::string(what) + ": " + cudaGetErrorString(e);
  if (e == cudaErrorNoDevice || e == cudaErrorInsufficientDriver) return PETIGA_CUDA_ERR_NODEVICE;
  if (e == cudaErrorMemoryAllocation) return PETIGA_CUDA_ERR_MEM;
  return PETIGA_CUDA_ERR_CUDA;
}

template <typename T>
static int upload(petiga_cuda_plan* P, const T* src, size_t n, T** dst) {
  *dst = nullptr;
  if (n == 0) n = 1;
  void* d = nullptr;
  PC_CUDA(cudaMalloc(&d, n * sizeof(T)));
  P->allocs.push_back(d);
  if (src) PC_CUDA(cudaMemcpyAsync(d, src, n * sizeof(T), cudaMemcpyHostToDevice, P->stream));
  *dst = static_cast<T*>(d);
  return 0;
}

// ---- pattern kernel: one warp per owned row, closed-form positions (IGACreateMat: petigamat.c:448-537) ----
struct PatParams {
  const int* rowG[3]; const int* W[3]; const uint32_t* seg[3]; const int* first[3]; const int* own[3];
  const int* box_ls[3]; const int* box_lw[3]; const int* rank_start; const int64_t* rowbase;
  int gs[3], nnp[3], Pn[3];
  int nown, bs;
  int* colidx;
};

__global__ void pattern_kernel(const __grid_constant__ PatParams pp) {
  const int warps_per_block = blockDim.x / 32, lane = threadIdx.x & 31;
  for (int row = blockIdx.x * warps_per_block + threadIdx.x / 32; row < pp.nown; row += gridDim.x * warps_per_block) {
    int node[3], g[3], W[3];
#pragma unroll
    for (int d = 0; d < 3; d++) { node[d] = pp.rowG[d][row]; g[d] = node[d] - pp.gs[d]; W[d] = pp.W[d][g[d]]; }
    const int nw = W[0] * W[1] * W[2];
    const int64_t base = pp.rowbase[row];
    for (int e = lane; e < nw; e += 32) {
      int c[3] = {e % W[0], (e / W[0]) % W[1], e / (W[0] * W[1])};
      int B[3], S[3], Lc[3], gid_r[3], w[3];
#pragma unroll
      for (int d = 0; d < 3; d++) {
        uint32_t s = pp.seg[d][g[d] * kMaxW + c[d]];
        B[d] = s & 255; S[d] = (s >> 8) & 255; Lc[d] = (s >> 16) & 255;
        int cc = pp.first[d][node[d]] + c[d];
        w[d] = cc < 0 ? pp.nnp[d] + cc : (cc >= pp.nnp[d] ? cc % pp.nnp[d] : cc);
        gid_r[d] = pp.own[d][w[d]];
      }
      int pos = B[2] * W[1] * W[0] + S[2] * (B[1] * W[0] + S[1] * B[0]) + (Lc[2] * S[1] + Lc[1]) * S[0] + Lc[0];
      int q = gid_r[0] + pp.Pn[0] * (gid_r[1] + pp.Pn[1] * gid_r[2]);
      int l0 = pp.box_lw[0][gid_r[0]], l1 = pp.box_lw[1][gid_r[1]];
      int gid = pp.rank_start[q] + (w[0] - pp.box_ls[0][gid_r[0]]) + l0 * ((w[1] - pp.box_ls[1][gid_r[1]]) + l1 * (w[2] - pp.box_ls[2][gid_r[2]]));
      if (pp.bs == 1) pp.colidx[base + pos] = gid;
      else
        for (int r = 0; r < pp.bs; r++)
          for (int cc = 0; cc < pp.bs; cc++)
            pp.colidx[base * pp.bs * pp.bs + (int64_t)r * nw * pp.bs + (int64_t)pos * pp.bs + cc] = gid * pp.bs + cc;
    }
  }
}

__global__ void gather_owned_kernel(const double* __restrict__ src, double* __restrict__ dst, size_t n) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) dst[i] = src[i];
}

// BoundaryArea of an element face on a mapped geometry: sum over the face's quadrature points of the surface Jacobian
// sqrt|det(F F^T)|, F = d x / d(face parameters), times the weights (src/petigaelem.c:1132-1162 ->
// IGA_BoundaryArea_{2,3}D, src/petiga{2,3}d.F90; Rationalize + Jacobian there).  The rationalised sums are folded:
// F[r][s] = (Q[r][s] - S1[r] P[s] / W0) / W0 with W0 = sum W N0, S1 = sum W N1, P = sum W N0 X, Q = sum W N1 X.
template <int DIM>
__device__ double face_area_factor(const DevAxis* ax, const int* ID, int dir, int side, const double* __restrict__ X,
                                          const double* __restrict__ Wt) {
  if (DIM == 1) return 1.0;
  int fa[2] = {0, 0}, n = 0;
  for (int i = 0; i < DIM; i++) if (i != dir) fa[n++] = i;
  const int sd = DIM - 1;
  const DevAxis& A0 = ax[fa[0]];
  const DevAxis& A1 = ax[(sd > 1) ? fa[1] : fa[0]];
  const int ne0 = A0.nen, ne1 = (sd > 1) ? A1.nen : 1, nq0 = A0.nqp, nq1 = (sd > 1) ? A1.nqp : 1;
  const int kfix = side ? ax[dir].nen - 1 : 0;
  int g[3] = {0, 0, 0};
  g[dir] = ax[dir].offset[ID[dir]] + kfix - ax[dir].gs;
  const int b0 = A0.offset[ID[fa[0]]] - A0.gs, b1 = (sd > 1) ? A1.offset[ID[fa[1]]] - A1.gs : 0;
  double dS = 0.0;
  for (int jq = 0; jq < nq1; jq++)
    for (int iq = 0; iq < nq0; iq++) {
      double W0 = 0.0, S1[2] = {0, 0}, P[3] = {0, 0, 0}, Q[2][3] = {{0, 0, 0}, {0, 0, 0}};
      for (int ja = 0; ja < ne1; ja++) {
        const double j0 = (sd > 1) ? A1.value[((size_t)(ID[fa[1]] * nq1 + jq) * ne1 + ja) * 5] : 1.0;
        const double j1 = (sd > 1) ? A1.value[((size_t)(ID[fa[1]] * nq1 + jq) * ne1 + ja) * 5 + 1] : 0.0;
        if (sd > 1) g[fa[1]] = b1 + ja;
        for (int ia = 0; ia < ne0; ia++) {
          const double i0 = A0.value[((size_t)(ID[fa[0]] * nq0 + iq) * ne0 + ia) * 5];
          const double i1 = A0.value[((size_t)(ID[fa[0]] * nq0 + iq) * ne0 + ia) * 5 + 1];
          g[fa[0]] = b0 + ia;
          const int gidx = g[0] + ax[0].gw * (g[1] + ax[1].gw * g[2]);
          const double w = Wt ? Wt[gidx] : 1.0;
          const double N0 = w * i0 * j0, N1a = w * i1 * j0, N1b = w * i0 * j1;
          W0 += N0; S1[0] += N1a; S1[1] += N1b;
#pragma unroll
          for (int s = 0; s < DIM; s++) {
            const double x = X[(size_t)gidx * DIM + s];
            P[s] = fma(N0, x, P[s]); Q[0][s] = fma(N1a, x, Q[0][s]); Q[1][s] = fma(N1b, x, Q[1][s]);
          }
        }
      }
      double F[2][3];
#pragma unroll
      for (int r = 0; r < 2; r++)
#pragma unroll
        for (int s = 0; s < DIM; s++) F[r][s] = Wt ? (Q[r][s] - S1[r] * P[s] / W0) / W0 : Q[r][s];
      double m00 = 0, m01 = 0, m11 = 0;
#pragma unroll
      for (int s = 0; s < DIM; s++) { m00 = fma(F[0][s], F[0][s], m00); m01 = fma(F[0][s], F[1][s], m01); m11 = fma(F[1][s], F[1][s], m11); }
      const double det = (sd > 1) ? m00 * m11 - m01 * m01 : m00;
      double wq = A0.weight[ID[fa[0]] * nq0 + iq];
      if (sd > 1) wq *= A1.weight[ID[fa[1]] * nq1 + jq];
      dS += sqrt(fabs(det)) * wq;
    }
  return dS;
}


struct FaceParams { DevAxis ax[3]; int dir, side, n0, n1; const double* X; const double* Wt; double* out; };

// one thread per element of the face (dir, side) inside this rank's element box; kept out of the assembly kernels so that
// the rare mapped-load case does not cost them registers (122 vs 77 in quad_sf_kernel<3,3,1,4> when it was inlined)
template <int DIM>
__global__ void face_area_kernel(const __grid_constant__ FaceParams fp) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= fp.n0 * fp.n1) return;
  int fa[2] = {0, 0}, n = 0;
  for (int i = 0; i < DIM; i++) if (i != fp.dir) fa[n++] = i;
  int ID[3] = {0, 0, 0};
  ID[fp.dir] = fp.side ? fp.ax[fp.dir].nel - 1 : 0;
  ID[fa[0]] = fp.ax[fa[0]].es + t % fp.n0;
  if (DIM > 2) ID[fa[1]] = fp.ax[fa[1]].es + t / fp.n0;
  fp.out[t] = face_area_factor<DIM>(fp.ax, ID, fp.dir, fp.side, fp.X, fp.Wt);
}

// IGASetFixTable: local-row vector -> ghost-box table [ghost box][dof] (the G2L scatter of src/petigaform.c IGASetFixTable)
__global__ void fixtable_scatter_kernel(const int* __restrict__ localrow, const double* __restrict__ loc, double* __restrict__ out, size_t ng, int dof) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < ng * dof; i += (size_t)gridDim.x * blockDim.x) {
    const size_t g = i / dof;
    out[i] = loc[(size_t)localrow[g] * dof + (i - g * dof)];
  }
}

// ||a - b||^2 and ||b||^2 over n doubles: per-CTA partial sums in a fixed order (deterministic), finished on the host.
// Used by the full-size parity tests to compare two 5.9 GB value arrays without moving them off the device.
__global__ void __launch_bounds__(256) diff_norm_kernel(const double* __restrict__ a, const double* __restrict__ b, size_t n, double* __restrict__ part) {
  __shared__ double sd[8], sr[8];
  double d2 = 0.0, r2 = 0.0;
  const size_t chunk = (n + gridDim.x - 1) / gridDim.x, lo = (size_t)blockIdx.x * chunk, hi = lo + chunk < n ? lo + chunk : n;
  for (size_t i = lo + threadIdx.x; i < hi; i += 256) { const double x = a[i], y = b[i]; d2 = fma(x - y, x - y, d2); r2 = fma(y, y, r2); }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) { d2 += __shfl_xor_sync(0xffffffffu, d2, o); r2 += __shfl_xor_sync(0xffffffffu, r2, o); }
  if ((threadIdx.x & 31) == 0) { sd[threadIdx.x >> 5] = d2; sr[threadIdx.x >> 5] = r2; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double x = 0.0, y = 0.0;
    for (int w = 0; w < 8; w++) { x += sd[w]; y += sr[w]; }
    part[2 * blockIdx.x] = x; part[2 * blockIdx.x + 1] = y;
  }
}

// FP64 FMA peak: 8 independent DFMA chains per thread, 4 CTAs of 256 threads per SM (the roofline denominator of the
// quadrature kernels; MEASURED_PEAKS.json carries no FP64 figure, SURVEY 8d asks for a measured one)
__global__ void __launch_bounds__(256) dfma_peak_kernel(double* out, int iters, double a, double b) {
  double x0 = threadIdx.x, x1 = x0 + 1, x2 = x0 + 2, x3 = x0 + 3, x4 = x0 + 4, x5 = x0 + 5, x6 = x0 + 6, x7 = x0 + 7;
  for (int i = 0; i < iters; i++) {
#pragma unroll
    for (int k = 0; k < 8; k++) {
      x0 = fma(x0, a, b); x1 = fma(x1, a, b); x2 = fma(x2, a, b); x3 = fma(x3, a, b);
      x4 = fma(x4, a, b); x5 = fma(x5, a, b); x6 = fma(x6, a, b); x7 = fma(x7, a, b);
    }
  }
  const double s = ((x0 + x1) + (x2 + x3)) + ((x4 + x5) + (x6 + x7));
  if (s == 12345.678) out[0] = s;   // never true for the arguments used; keeps the chains alive
}

void fill_fix_sides(const petiga_cuda_plan* P, bool loads, FixSide out[3][2]) {
  if (!P->has_bc) return;
  const Layout& L = P->L;
  for (int d = 0; d < L.dim; d++)
    for (int s = 0; s < 2; s++) {
      FixSide& fs = out[d][s];
      for (int k = 0; k < P->bc.vcount[d][s]; k++) {
        const int c = P->bc.vfield[d][s][k];
        if (c >= L.dof || fs.vcount >= kMaxDof) continue;   // AddFixa skips fields >= dof (petigaelem.c:1179)
        fs.vfield[fs.vcount] = c; fs.vvalue[fs.vcount] = P->bc.vvalue[d][s][k]; fs.vcount++;
      }
      for (int k = 0; loads && k < P->bc.lcount[d][s]; k++) {
        const int c = P->bc.lfield[d][s][k];
        if (c >= L.dof || fs.lcount >= kMaxDof) continue;
        fs.lfield[fs.lcount] = c; fs.lvalue[fs.lcount] = P->bc.lvalue[d][s][k]; fs.lcount++;
      }
    }
}

}  // namespace pc

using namespace pc;

extern "C" {

int petiga_cuda_version(void) { return PETIGA_CUDA_VERSION; }

const char* petiga_cuda_strerror(int code) {
  switch (code) {
    case PETIGA_CUDA_OK: return "success";
    case PETIGA_CUDA_ERR_ARG: return "invalid argument";
    case PETIGA_CUDA_ERR_ORDER: return "operation called out of order";
    case PETIGA_CUDA_ERR_SUP: return "configuration not supported by the device path";
    case PETIGA_CUDA_ERR_MEM: return "out of memory";
    case PETIGA_CUDA_ERR_CUDA: return "CUDA runtime error";
    case PETIGA_CUDA_ERR_NODEVICE: return "no CUDA device (libpetiga_cuda has no CPU fallback)";
    case PETIGA_CUDA_ERR_NCCL: return "NCCL error";
  }
  return "unknown error";
}

const char* petiga_cuda_last_error(void) { return g_last_error.c_str(); }

int petiga_cuda_device_count(int* count) {
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (count) *count = (e == cudaSuccess) ? n : 0;
  if (e != cudaSuccess) return cuda_fail(e, "cudaGetDeviceCount");
  return n > 0 ? 0 : PETIGA_CUDA_ERR_NODEVICE;
}

int petiga_cuda_plan_create(petiga_cuda_plan** plan, const petiga_cuda_space* sp, int rank, int nranks, void* nccl_comm,
                            void* stream, int device) {
  if (!plan || !sp) return PETIGA_CUDA_ERR_ARG;
  *plan = nullptr;
  int ndev = 0;
  int rc = petiga_cuda_device_count(&ndev);
  if (rc) { if (g_last_error.empty()) set_error("no CUDA device; libpetiga_cuda has no CPU fallback"); return rc; }
  if (device < 0 || device >= ndev) { set_error("bad device ordinal"); return PETIGA_CUDA_ERR_ARG; }
  petiga_cuda_plan* P = new (std::nothrow) petiga_cuda_plan();
  if (!P) return PETIGA_CUDA_ERR_MEM;
  memset(&P->bc, 0, sizeof(P->bc));
  rc = build_layout(*sp, rank, nranks, P->L);
  if (rc) { set_error(P->L.error); delete P; return rc; }
  if (sp->order < 1 || sp->order > 4) { set_error("order must be in [1,4]"); delete P; return PETIGA_CUDA_ERR_ARG; }
  P->order = sp->order;
  P->device = device;
  P->nccl = nccl_comm;
  auto bail = [&](int code) { petiga_cuda_plan_destroy(P); return code; };
  if (cudaSetDevice(device) != cudaSuccess) return bail(cuda_fail(cudaGetLastError(), "cudaSetDevice"));
  if (stream) P->stream = (cudaStream_t)stream;
  else {
    cudaError_t e = cudaStreamCreateWithFlags(&P->stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) return bail(cuda_fail(e, "cudaStreamCreate"));
    P->own_stream = true;
  }
  cudaDeviceGetAttribute(&P->num_sms, cudaDevAttrMultiProcessorCount, device);
  cudaEventCreate(&P->ev0);
  cudaEventCreate(&P->ev1);
  const Layout& L = P->L;
  for (int d = 0; d < 3; d++) {
    const AxisLayout& a = L.ax[d];
    DevAxis& da = P->dax[d];
    const size_t nq = (size_t)a.nel * a.nqp;
    if (!sp->value[d] || !sp->weight[d] || !sp->point[d] || !sp->detJac[d]) { set_error("missing basis tables"); return bail(PETIGA_CUDA_ERR_ARG); }
    double *v, *w, *pt, *dj; int *off, *W, *lo, *simp; uint32_t* seg;
    if ((rc = upload(P, sp->value[d], nq * (a.p + 1) * 5, &v))) return bail(rc);
    if ((rc = upload(P, sp->weight[d], nq, &w))) return bail(rc);
    if ((rc = upload(P, sp->point[d], nq, &pt))) return bail(rc);
    if ((rc = upload(P, sp->detJac[d], (size_t)a.nel, &dj))) return bail(rc);
    if ((rc = upload(P, sp->offset[d], (size_t)a.nel, &off))) return bail(rc);
    if ((rc = upload(P, a.W.data(), a.W.size(), &W))) return bail(rc);
    if ((rc = upload(P, a.lo.data(), a.lo.size(), &lo))) return bail(rc);
    if ((rc = upload(P, a.seg.data(), a.seg.size(), &seg))) return bail(rc);
    if ((rc = upload(P, a.simple.data(), a.simple.size(), &simp))) return bail(rc);
    da.value = v; da.weight = w; da.point = pt; da.detJac = dj; da.offset = off; da.W = W; da.lo = lo; da.seg = seg; da.simple = simp;
    da.nel = a.nel; da.nqp = a.nqp; da.nen = a.p + 1; da.p = a.p; da.gs = a.gs; da.gw = a.gw; da.es = a.es; da.ew = a.ew;
    da.periodic = a.periodic; da.nnp = a.nnp;
    P->detJac_h[d].assign(sp->detJac[d], sp->detJac[d] + a.nel);
    if ((rc = upload(P, L.rowG[d].data(), L.rowG[d].size(), &P->d_rowG[d]))) return bail(rc);
    if ((rc = upload(P, a.first.data(), a.first.size(), &P->d_first[d]))) return bail(rc);
    if ((rc = upload(P, a.own.data(), a.own.size(), &P->d_own[d]))) return bail(rc);
    if ((rc = upload(P, a.box_ls.data(), a.box_ls.size(), &P->d_box_ls[d]))) return bail(rc);
    if ((rc = upload(P, a.box_lw.data(), a.box_lw.size(), &P->d_box_lw[d]))) return bail(rc);
  }
  if ((rc = upload(P, L.localrow.data(), L.localrow.size(), &P->d_localrow))) return bail(rc);
  if ((rc = upload(P, L.rowbase.data(), L.rowbase.size(), &P->d_rowbase))) return bail(rc);
  if ((rc = upload(P, L.rank_start.data(), L.rank_start.size(), &P->d_rank_start))) return bail(rc);
  if (L.nranks > 1) {
    const size_t nl = (size_t)L.nloc * L.dof;
    if ((rc = upload<double>(P, nullptr, nl, &P->d_rhs_loc))) return bail(rc);
    if ((rc = upload<double>(P, nullptr, nl, &P->d_U_loc))) return bail(rc);
    if ((rc = upload<double>(P, nullptr, nl, &P->d_V_loc))) return bail(rc);
    if ((rc = upload<double>(P, nullptr, nl, &P->d_W_loc))) return bail(rc);
    std::vector<int> rows;
    std::vector<int64_t> offs;      // prefix sum of the row lengths inside each peer's slab (the sender packs rows back to back)
    P->recv_row_off.clear();
    for (auto& r : L.recv) {
      P->recv_row_off.push_back(rows.size());
      rows.insert(rows.end(), r.rows.begin(), r.rows.end());
      int64_t o = 0;
      for (int row : r.rows) { offs.push_back(o); o += L.rowbase[row + 1] - L.rowbase[row]; }
    }
    P->recv_row_off.push_back(rows.size());
    if ((rc = upload(P, rows.data(), rows.size(), &P->d_recv_rows))) return bail(rc);
    if ((rc = upload(P, offs.data(), offs.size(), &P->d_recv_off))) return bail(rc);
  }
  cudaError_t e = cudaStreamSynchronize(P->stream);
  if (e != cudaSuccess) return bail(cuda_fail(e, "plan upload"));
  *plan = P;
  return 0;
}

int petiga_cuda_plan_destroy(petiga_cuda_plan* P) {
  if (!P) return 0;
  cudaSetDevice(P->device);
  if (P->stream) cudaStreamSynchronize(P->stream);
  for (void* d : P->allocs) cudaFree(d);
  for (int b = 0; b < 2; b++) { cudaFree(P->d_rowptr[b]); cudaFree(P->d_colidx[b]); }
  cudaFree(P->d_X); cudaFree(P->d_W); cudaFree(P->d_fixtable); cudaFree(P->d_ghost_values); cudaFree(P->d_recv);
  cudaFree(P->d_scalar); cudaFree(P->d_sf3_dprime); cudaFree(P->d_solve_work); cudaFree(P->d_solve_xfull); cudaFree(P->d_gmres_work); cudaFree(P->d_values_own); cudaFree(P->d_rhs_own); cudaFree(P->d_U_own); cudaFree(P->d_V_own);
  if (P->h_pinned) cudaFreeHost(P->h_pinned);
  if (P->ev0) cudaEventDestroy(P->ev0);
  if (P->ev1) cudaEventDestroy(P->ev1);
  if (P->own_stream && P->stream) cudaStreamDestroy(P->stream);
  delete P;
  return 0;
}

int petiga_cuda_set_option(petiga_cuda_plan* P, const char* name, double value) {
  if (!P || !name) return PETIGA_CUDA_ERR_ARG;
  if (!strcmp(name, "path")) { int v = (int)value; if (v < 0 || v > 2) return PETIGA_CUDA_ERR_ARG; P->path = v; return 0; }
  if (!strcmp(name, "scatter")) { P->scatter = (int)value; return 0; }
  if (!strcmp(name, "quad_impl")) { int v = (int)value; if (v < -1 || v > 3) return PETIGA_CUDA_ERR_ARG; P->quad_impl = v; return 0; }
  if (!strcmp(name, "kron_minb_rows")) { P->kron_minb_rows = (int)value; P->config_version++; return 0; }
  if (!strcmp(name, "kron_bulk")) { P->kron_bulk = value != 0; P->config_version++; return 0; }
  if (!strcmp(name, "sf3_static")) { P->sf3_static = value != 0; return 0; }
  if (!strcmp(name, "sf3_variant")) { int v = (int)value; if (v < 0 || v > 1) return PETIGA_CUDA_ERR_ARG; P->sf3_variant = v; return 0; }
  set_error(std::string("unknown option ") + name);
  return PETIGA_CUDA_ERR_ARG;
}

int petiga_cuda_get_stat(petiga_cuda_plan* P, const char* name, double* value) {
  if (!P || !name || !value) return PETIGA_CUDA_ERR_ARG;
  if (!strcmp(name, "launches")) { *value = (double)P->launches; return 0; }
  if (!strcmp(name, "last_path")) { *value = (double)P->last_path; return 0; }
  if (!strcmp(name, "last_impl")) { *value = (double)P->last_impl; return 0; }
  if (!strcmp(name, "last_sf3_static")) { *value = (double)P->last_sf3_static; return 0; }
  if (!strcmp(name, "last_sf3_variant")) { *value = (double)P->last_sf3_variant; return 0; }
  if (!strcmp(name, "last_kernel_ms")) { *value = P->last_kernel_ms; return 0; }
  if (!strcmp(name, "last_flops")) { *value = P->last_flops; return 0; }
  if (!strcmp(name, "num_sms")) { *value = P->num_sms; return 0; }
  if (!strcmp(name, "nghostrows")) { *value = P->L.nghostrows; return 0; }
  if (!strcmp(name, "nnz_loc")) { *value = (double)P->L.nnz_loc; return 0; }
  return PETIGA_CUDA_ERR_ARG;
}

int petiga_cuda_set_geometry(petiga_cuda_plan* P, int nsd, const double* X, const double* W) {
  if (!P) return PETIGA_CUDA_ERR_ARG;
  PC_CUDA(cudaSetDevice(P->device));
  PC_CUDA(cudaStreamSynchronize(P->stream));
  cudaFree(P->d_X); cudaFree(P->d_W);
  P->d_X = P->d_W = nullptr;
  P->config_version++;
  if (!X) return 0;
  if (nsd != P->L.dim) { set_error("geometry: nsd must equal dim on the device path (manifolds unsupported)"); return PETIGA_CUDA_ERR_SUP; }
  const size_t ng = P->L.localrow.size();
  PC_CUDA(cudaMalloc(&P->d_X, ng * nsd * sizeof(double)));
  PC_CUDA(cudaMemcpy(P->d_X, X, ng * nsd * sizeof(double), cudaMemcpyHostToDevice));
  if (W) {
    PC_CUDA(cudaMalloc(&P->d_W, ng * sizeof(double)));
    PC_CUDA(cudaMemcpy(P->d_W, W, ng * sizeof(double), cudaMemcpyHostToDevice));
  }
  return 0;
}

int petiga_cuda_set_bc(petiga_cuda_plan* P, const petiga_cuda_bc* bc) {
  if (!P) return PETIGA_CUDA_ERR_ARG;
  PC_CUDA(cudaSetDevice(P->device));
  PC_CUDA(cudaStreamSynchronize(P->stream));
  cudaFree(P->d_fixtable);
  P->d_fixtable = nullptr;
  P->has_bc = false;
  P->config_version++;
  memset(&P->bc, 0, sizeof(P->bc));
  if (!bc) return 0;
  for (int d = 0; d < 3; d++)
    for (int s = 0; s < 2; s++) {
      if (bc->vcount[d][s] < 0 || bc->vcount[d][s] > 64 || bc->lcount[d][s] < 0 || bc->lcount[d][s] > 64) return PETIGA_CUDA_ERR_ARG;
      if (d < P->L.dim && (bc->vcount[d][s] || bc->lcount[d][s])) P->has_bc = true;
    }
  // copy with the semantics of IGAFormSetBoundaryValue/Load (src/petigaform.c:102-149): one entry per field, a repeated field
  // overwrites the earlier value; negative fields are an argument error (PETSC_ERR_ARG_OUTOFRANGE there)
  for (int d = 0; d < 3; d++)
    for (int s = 0; s < 2; s++) {
      for (int k = 0; k < bc->vcount[d][s]; k++) {
        const int f = bc->vfield[d][s][k];
        if (f < 0) { memset(&P->bc, 0, sizeof(P->bc)); P->has_bc = false; set_error("set_bc: negative field index"); return PETIGA_CUDA_ERR_ARG; }
        int pos = -1;
        for (int j = 0; j < P->bc.vcount[d][s]; j++) if (P->bc.vfield[d][s][j] == f) pos = j;
        if (pos < 0) pos = P->bc.vcount[d][s]++;
        P->bc.vfield[d][s][pos] = f; P->bc.vvalue[d][s][pos] = bc->vvalue[d][s][k];
      }
      for (int k = 0; k < bc->lcount[d][s]; k++) {
        const int f = bc->lfield[d][s][k];
        if (f < 0) { memset(&P->bc, 0, sizeof(P->bc)); P->has_bc = false; set_error("set_bc: negative field index"); return PETIGA_CUDA_ERR_ARG; }
        int pos = -1;
        for (int j = 0; j < P->bc.lcount[d][s]; j++) if (P->bc.lfield[d][s][j] == f) pos = j;
        if (pos < 0) pos = P->bc.lcount[d][s]++;
        P->bc.lfield[d][s][pos] = f; P->bc.lvalue[d][s][pos] = bc->lvalue[d][s][k];
      }
    }
  P->bc.fixtableU = nullptr;
  if (bc->fixtableU) {
    const size_t n = P->L.localrow.size() * P->L.dof;
    PC_CUDA(cudaMalloc(&P->d_fixtable, n * sizeof(double)));
    PC_CUDA(cudaMemcpy(P->d_fixtable, bc->fixtableU, n * sizeof(double), cudaMemcpyHostToDevice));
  }
  return 0;
}

int petiga_cuda_set_fixtable_device(petiga_cuda_plan* P, const double* table_own) {
  if (!P) return PETIGA_CUDA_ERR_ARG;
  if (P->L.collocation && table_own) { set_error("set_fixtable_device: IGASetFixTable is not supported on a collocation plan"); return PETIGA_CUDA_ERR_SUP; }
  PC_CUDA(cudaSetDevice(P->device));
  PC_CUDA(cudaStreamSynchronize(P->stream));
  cudaFree(P->d_fixtable);
  P->d_fixtable = nullptr;
  P->config_version++;
  if (!table_own) return 0;
  const Layout& L = P->L;
  const size_t ng = L.localrow.size();
  PC_CUDA(cudaMalloc(&P->d_fixtable, ng * L.dof * sizeof(double)));
  const double* loc = table_own;          // one rank: local rows == owned rows
  double* tmp = nullptr;
  if (L.nranks > 1) {                     // ghost nodes carry their owner's table value (VecScatter g2l)
    PC_CUDA(cudaMalloc(&tmp, (size_t)L.nloc * L.dof * sizeof(double)));
    int rc = halo_state(P, table_own, tmp);
    if (rc) { cudaFree(tmp); return rc; }
    loc = tmp;
  }
  const int blocks = (int)std::min<size_t>((ng * L.dof + 255) / 256, (size_t)P->num_sms * 8);
  fixtable_scatter_kernel<<<std::max(blocks, 1), 256, 0, P->stream>>>(P->d_localrow, loc, P->d_fixtable, ng, L.dof);
  PC_CUDA(cudaGetLastError());
  P->launches++;
  PC_CUDA(cudaStreamSynchronize(P->stream));
  cudaFree(tmp);
  return 0;
}

int petiga_cuda_form_select(petiga_cuda_plan* P, int slot, int form_id, const double* params, int nparams) {
  if (P && slot >= 0 && slot < PETIGA_NSLOTS && form_id == -1) {   // IGASetForm*(iga, NULL, NULL): the slot has no callback any more
    P->slots[slot].form = -1;
    P->config_version++;
    return 0;
  }
  if (!P || slot < 0 || slot >= PETIGA_NSLOTS || form_id < 0 || form_id >= PETIGA_NFORMS || nparams < 0 || nparams > kMaxPrm) {
    set_error("form_select: bad slot / form / nparams");
    return PETIGA_CUDA_ERR_ARG;
  }
  FormInfo fi = form_info(form_id, slot, P->L.dim, P->L.dof);
  if (!fi.valid) { set_error("form_select: this built-in form does not provide that slot for this dim/dof (PETSC_ERR_SUP)"); return PETIGA_CUDA_ERR_SUP; }
  P->slots[slot].form = form_id;
  P->config_version++;
  memset(P->slots[slot].prm, 0, sizeof(P->slots[slot].prm));
  for (int k = 0; k < nparams; k++) P->slots[slot].prm[k] = params[k];
  return 0;
}

int petiga_cuda_plan_sizes(petiga_cuda_plan* P, int* nown, int* nghost, int64_t* nnzb) {
  if (!P) return PETIGA_CUDA_ERR_ARG;
  if (nown) *nown = P->L.nown;
  if (nghost) *nghost = (int)P->L.localrow.size();
  if (nnzb) *nnzb = P->L.nnz_own;
  return 0;
}

int petiga_cuda_plan_lgmap_host(petiga_cuda_plan* P, int* lgmap) {
  if (!P || !lgmap) return PETIGA_CUDA_ERR_ARG;
  memcpy(lgmap, P->L.lgmap.data(), P->L.lgmap.size() * sizeof(int));
  return 0;
}

int petiga_cuda_plan_pattern(petiga_cuda_plan* P, int block, int* nrows, int64_t* nnz, const int** d_rowptr, const int** d_colidx) {
  if (!P || (block != 0 && block != 1)) return PETIGA_CUDA_ERR_ARG;
  const Layout& L = P->L;
  const int bs = block ? 1 : L.dof;
  const int64_t n = L.nnz_own * bs * bs;
  if (n > INT32_MAX) { set_error("pattern: more than 2^31-1 nonzeros on one rank; use the block (BAIJ) layout or more ranks"); return PETIGA_CUDA_ERR_SUP; }
  PC_CUDA(cudaSetDevice(P->device));
  if (!P->d_rowptr[block]) {
    std::vector<int> rp((size_t)L.nown * bs + 1);
    rp[0] = 0;
    for (int r = 0; r < L.nown; r++) {
      int W = L.rowW[0][r] * L.rowW[1][r] * L.rowW[2][r];
      for (int k = 0; k < bs; k++) rp[(size_t)r * bs + k + 1] = (int)(L.rowbase[r] * bs * bs + (int64_t)(k + 1) * W * bs);
    }
    PC_CUDA(cudaMalloc(&P->d_rowptr[block], rp.size() * sizeof(int)));
    PC_CUDA(cudaMemcpyAsync(P->d_rowptr[block], rp.data(), rp.size() * sizeof(int), cudaMemcpyHostToDevice, P->stream));
    PC_CUDA(cudaMalloc(&P->d_colidx[block], (size_t)(n > 0 ? n : 1) * sizeof(int)));
    PatParams pp;
    for (int d = 0; d < 3; d++) {
      pp.rowG[d] = P->d_rowG[d]; pp.W[d] = P->dax[d].W; pp.seg[d] = P->dax[d].seg; pp.first[d] = P->d_first[d]; pp.own[d] = P->d_own[d];
      pp.box_ls[d] = P->d_box_ls[d]; pp.box_lw[d] = P->d_box_lw[d]; pp.gs[d] = L.ax[d].gs; pp.nnp[d] = L.ax[d].nnp; pp.Pn[d] = L.ax[d].P;
    }
    pp.rank_start = P->d_rank_start; pp.rowbase = P->d_rowbase; pp.nown = L.nown; pp.bs = bs; pp.colidx = P->d_colidx[block];
    const int blocks = std::max(1, std::min((L.nown + 7) / 8, P->num_sms * 16));
    pattern_kernel<<<blocks, 256, 0, P->stream>>>(pp);
    PC_CUDA(cudaGetLastError());
    P->launches++;
    PC_CUDA(cudaStreamSynchronize(P->stream));
  }
  if (nrows) *nrows = L.nown * bs;
  if (nnz) *nnz = n;
  if (d_rowptr) *d_rowptr = P->d_rowptr[block];
  if (d_colidx) *d_colidx = P->d_colidx[block];
  return 0;
}

int petiga_cuda_plan_pattern_host(petiga_cuda_plan* P, int block, int* rowptr, int* colidx) {
  int nrows = 0; int64_t nnz = 0; const int *drp, *dci;
  int rc = petiga_cuda_plan_pattern(P, block, &nrows, &nnz, &drp, &dci);
  if (rc) return rc;
  if (rowptr) PC_CUDA(cudaMemcpy(rowptr, drp, ((size_t)nrows + 1) * sizeof(int), cudaMemcpyDeviceToHost));
  if (colidx) PC_CUDA(cudaMemcpy(colidx, dci, (size_t)nnz * sizeof(int), cudaMemcpyDeviceToHost));
  return 0;
}

// ---------------------------------------------------------------------------------------------
static int ensure(double** buf, size_t* cap, size_t n) {
  if (*cap >= n && *buf) return 0;
  cudaFree(*buf);
  *buf = nullptr; *cap = 0;
  PC_CUDA(cudaMalloc(buf, (n ? n : 1) * sizeof(double)));
  *cap = n;
  return 0;
}

int petiga_cuda_compute(petiga_cuda_plan* P, int slot, int block, double shift, const double* V, double t, const double* U,
                        double* values, double* rhs) {
  return petiga_cuda_compute_ext(P, slot, block, shift, V, t, U, 0.0, nullptr, 0.0, values, rhs);
}

int petiga_cuda_compute_ext(petiga_cuda_plan* P, int slot, int block, double shift, const double* V, double t, const double* U,
                            double shift2, const double* W, double t0, double* values, double* rhs) {
  if (!P || slot < 0 || slot >= PETIGA_NSLOTS || (block != 0 && block != 1)) return PETIGA_CUDA_ERR_ARG;
  const Layout& L = P->L;
  const int form = P->slots[slot].form;
  if (form < 0) { set_error("compute: no form selected for this slot (IGACheckFormOp)"); return PETIGA_CUDA_ERR_ORDER; }
  FormInfo fi = form_info(form, slot, L.dim, L.dof);
  if (!fi.valid) return PETIGA_CUDA_ERR_SUP;
  const bool want_mat = slot_has_mat(slot), want_vec = slot_has_vec(slot);
  const bool state = slot_has_state(slot), has_v = slot_has_v(slot), has_w = slot_has_w(slot);
  if (want_mat && !values) { set_error("compute: values == NULL"); return PETIGA_CUDA_ERR_ARG; }
  if (want_vec && !rhs) { set_error("compute: rhs == NULL"); return PETIGA_CUDA_ERR_ARG; }
  if (state && !U) { set_error("compute: U == NULL"); return PETIGA_CUDA_ERR_ARG; }
  if (has_v && !V) { set_error("compute: V == NULL"); return PETIGA_CUDA_ERR_ARG; }
  if (has_w && !W) { set_error("compute: the third vector (U0 / A) == NULL"); return PETIGA_CUDA_ERR_ARG; }
  if (fi.order > P->order) { set_error("compute: form reads derivatives above IGASetOrder"); return PETIGA_CUDA_ERR_ARG; }
  if (L.collocation || fi.colloc) {   // isogeometric collocation: its own kernel, nothing else runs on such a plan
    if (!L.collocation) { set_error("compute: a collocation form needs a collocation plan (IGASetUseCollocation)"); return PETIGA_CUDA_ERR_SUP; }
    if (!fi.colloc) { set_error("compute: a collocation plan runs the collocation forms only (IGADeviceForm_*Collocation)"); return PETIGA_CUDA_ERR_SUP; }
    if (P->path == PETIGA_PATH_KRONECKER) { set_error("compute: the separable path does not apply to collocation"); return PETIGA_CUDA_ERR_SUP; }
    for (int d = 0; d < L.dim; d++)
      for (int s = 0; s < 2; s++) {
        if (P->visit[d][s]) { set_error("compute: IGASetBoundaryForm is not supported with collocation"); return PETIGA_CUDA_ERR_SUP; }
        if (P->has_bc && P->bc.lcount[d][s]) { set_error("compute: IGASetBoundaryLoad is not supported with collocation"); return PETIGA_CUDA_ERR_SUP; }
      }
    if (P->d_fixtable) { set_error("compute: IGASetFixTable is not supported with collocation"); return PETIGA_CUDA_ERR_SUP; }
    PC_CUDA(cudaSetDevice(P->device));
    nvtx_push(slot);
    cudaEventRecord(P->ev0, P->stream);
    const int rc = launch_collocation(P, slot, form, values, rhs);
    cudaEventRecord(P->ev1, P->stream);
    nvtx_pop();
    if (rc) return rc;
    P->last_path = PETIGA_PATH_COLLOCATION;
    P->last_impl = -1;
    P->last_flops = 0;
    return 0;
  }
  PC_CUDA(cudaSetDevice(P->device));
  const int bs2 = L.dof * L.dof;
  const size_t nval = (size_t)L.nnz_own * bs2, nvec = (size_t)L.nown * L.dof;
  const bool multi = L.nranks > 1;
  nvtx_push(slot);

  // boundary-integral pass (IGASetBoundaryForm): which faces are visited, and does the form have a face term?
  bool any_visit = false;
  for (int d = 0; d < L.dim; d++) for (int s = 0; s < 2; s++) if (P->visit[d][s] && !L.ax[d].periodic) any_visit = true;
  if (any_visit && !(fi.bnd_mat || fi.bnd_vec)) { nvtx_pop(); set_error("compute: a face is enabled with IGASetBoundaryForm but this built-in form has no boundary term"); return PETIGA_CUDA_ERR_SUP; }
  const bool bnd_pass = any_visit && ((want_vec && fi.bnd_vec) || (want_mat && fi.bnd_mat));
  // path selection
  const bool kron_ok = kron_applicable(P, slot, form) && !bnd_pass;
  if (P->path == PETIGA_PATH_KRONECKER && !kron_ok) { nvtx_pop(); set_error("compute: separable path not applicable (geometry, state or non-separable form)"); return PETIGA_CUDA_ERR_SUP; }
  const bool use_kron = kron_ok && P->path != PETIGA_PATH_QUADRATURE;
  P->last_path = use_kron ? PETIGA_PATH_KRONECKER : PETIGA_PATH_QUADRATURE;
  P->last_flops = 0;
  struct Pop { ~Pop() { nvtx_pop(); } } pop_on_exit;

  cudaEventRecord(P->ev0, P->stream);
  bool quad_mat = want_mat;   // does the quadrature kernel still have to produce the matrix?
  if (use_kron) {   // write-once path: no zeroing, no atomics, no exchange
    const bool hybrid = want_vec && !fi.constant_f;   // e.g. L2Projection: separable mass matrix, point-wise load f(x)
    int rc = launch_kronecker(P, slot, block, want_mat ? values : nullptr, (want_vec && !hybrid) ? rhs : nullptr);
    if (rc || !hybrid) { cudaEventRecord(P->ev1, P->stream); return rc; }
    quad_mat = false;
  }

  // MatZeroEntries / VecZeroEntries (petigaksp.c:166-167)
  if (quad_mat) PC_CUDA(cudaMemsetAsync(values, 0, nval * sizeof(double), P->stream));
  double* rhs_k = rhs;
  if (multi) {
    if (quad_mat) {
      int rc = ensure(&P->d_ghost_values, &P->ghost_values_cap, (size_t)(L.nnz_loc - L.nnz_own) * bs2);
      if (rc) return rc;
      PC_CUDA(cudaMemsetAsync(P->d_ghost_values, 0, (size_t)(L.nnz_loc - L.nnz_own) * bs2 * sizeof(double), P->stream));
    }
    if (want_vec) { rhs_k = P->d_rhs_loc; PC_CUDA(cudaMemsetAsync(rhs_k, 0, (size_t)L.nloc * L.dof * sizeof(double), P->stream)); }
  } else if (want_vec) PC_CUDA(cudaMemsetAsync(rhs, 0, nvec * sizeof(double), P->stream));

  // IGAGetLocalVecArray: G2L halo of the state vectors (petigavec.c:256-269)
  const double *U_k = U, *V_k = V, *W_k = W;
  if (multi && state) {
    int rc = halo_state(P, U, P->d_U_loc);
    if (rc) return rc;
    U_k = P->d_U_loc;
    if (has_v) { rc = halo_state(P, V, P->d_V_loc); if (rc) return rc; V_k = P->d_V_loc; }
    if (has_w) { rc = halo_state(P, W, P->d_W_loc); if (rc) return rc; W_k = P->d_W_loc; }
  }

  KParams kp;
  memset(&kp, 0, sizeof(kp));
  for (int d = 0; d < 3; d++) kp.ax[d] = P->dax[d];
  kp.dim = L.dim; kp.dof = L.dof;
  kp.nelem = L.ax[0].ew * L.ax[1].ew * L.ax[2].ew;
  kp.nown = L.nown; kp.nnz_own = L.nnz_own;
  kp.localrow = P->d_localrow; kp.rowbase = P->d_rowbase;
  kp.values = values; kp.ghost_values = P->d_ghost_values; kp.rhs = rhs_k;
  kp.U = state ? U_k : nullptr; kp.V = has_v ? V_k : nullptr; kp.Wv = has_w ? W_k : nullptr;
  kp.shift2 = shift2; kp.t0 = t0;
  kp.face_axis = kp.face_side = -1;
  for (int d = 0; d < 3; d++) {
    kp.maxdeg = std::max(kp.maxdeg, d < L.dim ? L.ax[d].p : 0);
    for (int s2 = 0; s2 < 2; s2++) { kp.bnd_value[d][s2] = P->d_bnd_value[d][s2]; kp.bnd_point[d][s2] = P->bnd_point[d][s2]; }
  }
  kp.X = P->d_X; kp.Wt = P->d_W; kp.fixtable = P->d_fixtable;
  kp.any_bc = 0;
  const bool apply_bc = (slot != PETIGA_SLOT_VECTOR && slot != PETIGA_SLOT_MATRIX);   // IGAComputeVector/Matrix never fix (petigaksp.c:33-139)
  if (apply_bc) {
    fill_fix_sides(P, true, kp.bc);
    for (int d = 0; d < L.dim; d++)
      for (int s = 0; s < 2; s++) {
        const FixSide& fs = kp.bc[d][s];
        if (fs.vcount || fs.lcount) kp.any_bc = 1;   // periodic axes count too
        const int face_e = s ? L.ax[d].nel - 1 : 0;
        const bool touches = face_e >= L.ax[d].es && face_e < L.ax[d].es + L.ax[d].ew;   // only ranks whose element box reaches the face
        if (fs.lcount && P->d_X && L.dim > 1 && !L.ax[d].periodic && touches) {   // BoundaryArea on a mapped face (petigaelem.c:1132-1162)
          int fa[2] = {0, 0}, nfa = 0;
          for (int i = 0; i < L.dim; i++) if (i != d) fa[nfa++] = i;
          const int n0 = L.ax[fa[0]].ew, n1 = (L.dim > 2) ? L.ax[fa[1]].ew : 1;
          if (!P->d_face_dS[d][s]) {
            void* buf = nullptr;
            PC_CUDA(cudaMalloc(&buf, (size_t)n0 * n1 * sizeof(double)));
            P->allocs.push_back(buf);
            P->d_face_dS[d][s] = (double*)buf;
            P->face_version[d][s] = -1;
          }
          if (P->face_version[d][s] != P->config_version) {
            FaceParams fp;
            for (int i = 0; i < 3; i++) fp.ax[i] = P->dax[i];
            fp.dir = d; fp.side = s; fp.n0 = n0; fp.n1 = n1; fp.X = P->d_X; fp.Wt = P->d_W; fp.out = P->d_face_dS[d][s];
            const int nb = (n0 * n1 + 127) / 128;
            if (L.dim == 2) face_area_kernel<2><<<nb, 128, 0, P->stream>>>(fp);
            else face_area_kernel<3><<<nb, 128, 0, P->stream>>>(fp);
            PC_CUDA(cudaGetLastError());
            P->launches++;
            P->face_version[d][s] = P->config_version;
          }
          kp.face_dS[d][s] = P->d_face_dS[d][s];
        }
      }
  }
  kp.form = form; kp.slot = slot; kp.block = block;
  kp.mc0 = fi.mc0; kp.mc1 = quad_mat ? fi.mc1 : fi.mc0; kp.vc0 = fi.vc0; kp.vc1 = fi.vc1;
  kp.per_qp = fi.per_qp; kp.needs_x = fi.needs_x; kp.needs_state = fi.needs_state || (state && kp.any_bc);
  int c0 = 99, c1 = 0;
  if (kp.mc1 > kp.mc0) { c0 = std::min(c0, fi.mc0); c1 = std::max(c1, fi.mc1); }
  if (fi.vc1 > fi.vc0) { c0 = std::min(c0, fi.vc0); c1 = std::max(c1, fi.vc1); }
  if (c1 == 0) { c0 = 0; c1 = 1; }
  if (P->d_X) { c0 = 0; c1 = std::max(c1, 1 + L.dim); }
  if (kp.needs_state) c0 = std::min(c0, 0), c1 = std::max(c1, 1);
  kp.c0 = c0; kp.c1 = c1;
  memcpy(kp.prm, P->slots[slot].prm, sizeof(kp.prm));
  kp.shift = shift; kp.t = t;
  kp.noscatter = (P->scatter == 99);
  // kernel choice (measured, profiles/): the sum-factorised kernels win on large elements (3-D, p >= 2), the pair-loop kernel on
  // small ones where per-element set-up dominates (2-D p=2).  What the tuned kernels do not instantiate -- mixed degrees per
  // axis, degree > 4, dof > 3, second derivatives on mapped / NURBS geometry, the IE/RHS/I2 drivers -- runs the generic kernel.
  const bool need_gen = slot >= PETIGA_SLOT_IEFUNCTION || (P->d_X && fi.order > 1) || P->quad_impl == 2;
  int impl = P->quad_impl, rc;
  if (need_gen) { impl = 2; rc = launch_quadrature_gen(P, kp); }
  else {
    rc = PETIGA_CUDA_ERR_SUP;
    if (impl < 0 && kp.mc1 == kp.mc0) {   // no matrix to integrate (IGAComputeVector, or the separable path has written it): vector kernel
      rc = launch_quadrature_vec3(P, kp);
      if (rc == 0) impl = 4;
      else if (rc != PETIGA_CUDA_ERR_SUP) return rc;
    }
    if (rc == PETIGA_CUDA_ERR_SUP && (impl < 0 || impl == 3)) {   // third-generation kernel where it applies (3-D, p = 3, dof 1, constant-coefficient linear forms)
      rc = launch_quadrature_sf3(P, kp);
      if (rc == 0) impl = 3;
      else if (rc != PETIGA_CUDA_ERR_SUP || impl == 3) return rc;
    }
    if (rc == PETIGA_CUDA_ERR_SUP) {
      if (impl < 0) impl = (L.dim == 3 && L.ax[0].p >= 2) ? 0 : 1;
      rc = impl == 1 ? launch_quadrature(P, kp) : launch_quadrature_sf(P, kp);
    }
    if (rc == PETIGA_CUDA_ERR_SUP && P->quad_impl < 0) {
      impl = 1 - impl;
      rc = impl == 1 ? launch_quadrature(P, kp) : launch_quadrature_sf(P, kp);
      if (rc == PETIGA_CUDA_ERR_SUP) { impl = 2; rc = launch_quadrature_gen(P, kp); }
    }
  }
  if (rc) return rc;
  P->last_impl = impl;
  if (bnd_pass) {   // face terms go into the same (unified local) arrays, before the ghost-row exchange
    if (fi.bnd_mat) {   // full forms on the visited faces (matrix + vector terms): the generic kernel in face mode, one launch per face
      for (int d = 0; d < L.dim; d++)
        for (int s = 0; s < 2; s++) {
          if (!P->visit[d][s] || L.ax[d].periodic) continue;
          const int face_e = s ? L.ax[d].nel - 1 : 0;
          if (face_e < L.ax[d].es || face_e >= L.ax[d].es + L.ax[d].ew) continue;
          if (!P->d_bnd_value[d][s]) { set_error("compute: boundary tables not set (petiga_cuda_set_boundary_tables)"); return PETIGA_CUDA_ERR_ORDER; }
          KParams kf = kp;
          kf.face_axis = d; kf.face_side = s;
          kf.mc1 = want_mat ? fi.mc1 : fi.mc0;
          rc = launch_quadrature_gen(P, kf);
          if (rc) return rc;
        }
    } else {
      rc = launch_boundary_pass(P, slot, form, P->slots[slot].prm, rhs_k, apply_bc && P->has_bc);
      if (rc) return rc;
    }
  }
  cudaEventRecord(P->ev1, P->stream);
  if (multi) {
    rc = exchange_ghost_rows(P, block, values, rhs, quad_mat, want_vec);
    if (rc) return rc;
  }
  return 0;
}

int petiga_cuda_finish(petiga_cuda_plan* P) {
  if (!P) return PETIGA_CUDA_ERR_ARG;
  PC_CUDA(cudaSetDevice(P->device));
  PC_CUDA(cudaStreamSynchronize(P->stream));
  float ms = 0;
  if (cudaEventElapsedTime(&ms, P->ev0, P->ev1) == cudaSuccess) P->last_kernel_ms = ms;
  else (void)cudaGetLastError();
  return 0;
}

int petiga_cuda_compute_host(petiga_cuda_plan* P, int slot, int block, double shift, const double* V_host, double t,
                             const double* U_host, double* values_host, double* rhs_host) {
  if (!P) return PETIGA_CUDA_ERR_ARG;
  const Layout& L = P->L;
  PC_CUDA(cudaSetDevice(P->device));
  const size_t nval = (size_t)L.nnz_own * L.dof * L.dof, nvec = (size_t)L.nown * L.dof;
  size_t cap;
  if (values_host) { int rc = ensure(&P->d_values_own, &P->values_own_cap, nval); if (rc) return rc; }
  cap = P->d_rhs_own ? nvec : 0; { int rc = ensure(&P->d_rhs_own, &cap, nvec); if (rc) return rc; }
  if (U_host) { cap = P->d_U_own ? nvec : 0; int rc = ensure(&P->d_U_own, &cap, nvec); if (rc) return rc;
    PC_CUDA(cudaMemcpyAsync(P->d_U_own, U_host, nvec * sizeof(double), cudaMemcpyHostToDevice, P->stream)); }
  if (V_host) { cap = P->d_V_own ? nvec : 0; int rc = ensure(&P->d_V_own, &cap, nvec); if (rc) return rc;
    PC_CUDA(cudaMemcpyAsync(P->d_V_own, V_host, nvec * sizeof(double), cudaMemcpyHostToDevice, P->stream)); }
  int rc = petiga_cuda_compute(P, slot, block, shift, V_host ? P->d_V_own : nullptr, t, U_host ? P->d_U_own : nullptr,
                               values_host ? P->d_values_own : nullptr, rhs_host ? P->d_rhs_own : nullptr);
  if (rc) return rc;
  if (values_host) PC_CUDA(cudaMemcpyAsync(values_host, P->d_values_own, nval * sizeof(double), cudaMemcpyDeviceToHost, P->stream));
  if (rhs_host) PC_CUDA(cudaMemcpyAsync(rhs_host, P->d_rhs_own, nvec * sizeof(double), cudaMemcpyDeviceToHost, P->stream));
  return petiga_cuda_finish(P);
}

// ---- measured FP64 FMA peak of the device (roofline denominator for the quadrature kernels) ----
int petiga_cuda_measure_fp64(int device, double seconds, double* tflops_burst, double* tflops_sustained) {
  int ndev = 0;
  int rc = petiga_cuda_device_count(&ndev);
  if (rc) return rc;
  if (device < 0 || device >= ndev) return PETIGA_CUDA_ERR_ARG;
  PC_CUDA(cudaSetDevice(device));
  int sms = 0;
  PC_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
  double* d = nullptr;
  PC_CUDA(cudaMalloc(&d, 8));
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0); cudaEventCreate(&e1);
  const int blocks = sms * 4, iters = 4096;
  const double flop = 2.0 * 64.0 * iters * 256.0 * blocks;      // 64 DFMA per iteration per thread
  double best = 0.0, sus_flop = 0.0;
  float ms = 0.f;
  for (int it = 0; it < 12; it++) {   // burst: best single launch (~1 ms each)
    cudaEventRecord(e0);
    dfma_peak_kernel<<<blocks, 256>>>(d, iters, 0.999999, 1e-9);
    cudaEventRecord(e1);
    PC_CUDA(cudaEventSynchronize(e1));
    cudaEventElapsedTime(&ms, e0, e1);
    if (it >= 2 && ms > 0) best = std::max(best, flop / (ms * 1e-3) / 1e12);
  }
  // sustained: back-to-back launches for `seconds`
  const int nl = std::max(1, (int)(seconds * 1e3 / std::max(0.05, flop / (best * 1e12) * 1e3)));
  cudaEventRecord(e0);
  for (int it = 0; it < nl; it++) { dfma_peak_kernel<<<blocks, 256>>>(d, iters, 0.999999, 1e-9); sus_flop += flop; }
  cudaEventRecord(e1);
  PC_CUDA(cudaEventSynchronize(e1));
  cudaEventElapsedTime(&ms, e0, e1);
  PC_CUDA(cudaGetLastError());
  if (tflops_burst) *tflops_burst = best;
  if (tflops_sustained) *tflops_sustained = sus_flop / (ms * 1e-3) / 1e12;
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  cudaFree(d);
  return 0;
}

int petiga_cuda_diff_norm2(const double* d_a, const double* d_b, size_t n, double* diff2, double* ref2) {
  if (!d_a || !d_b || !diff2 || !ref2) return PETIGA_CUDA_ERR_ARG;
  const int blocks = 1184;
  double* part = nullptr;
  PC_CUDA(cudaMalloc(&part, 2 * blocks * sizeof(double)));
  diff_norm_kernel<<<blocks, 256>>>(d_a, d_b, n, part);
  std::vector<double> h(2 * blocks);
  cudaError_t e = cudaMemcpy(h.data(), part, h.size() * sizeof(double), cudaMemcpyDeviceToHost);
  cudaFree(part);
  if (e != cudaSuccess) return cuda_fail(e, "diff_norm2");
  double x = 0.0, y = 0.0;
  for (int b = 0; b < blocks; b++) { x += h[2 * b]; y += h[2 * b + 1]; }
  *diff2 = x; *ref2 = y;
  return 0;
}

// ---- small device-memory helpers (they act on the current device: call petiga_cuda_plan_activate first) ----
int petiga_cuda_plan_activate(petiga_cuda_plan* P) { if (!P) return PETIGA_CUDA_ERR_ARG; PC_CUDA(cudaSetDevice(P->device)); return 0; }
int petiga_cuda_malloc(void** ptr, size_t bytes) { if (!ptr) return PETIGA_CUDA_ERR_ARG; PC_CUDA(cudaMalloc(ptr, bytes ? bytes : 1)); return 0; }
int petiga_cuda_free(void* ptr) { PC_CUDA(cudaFree(ptr)); return 0; }
int petiga_cuda_memcpy_h2d(void* dst, const void* src, size_t bytes) { PC_CUDA(cudaMemcpy(dst, src, bytes, cudaMemcpyHostToDevice)); return 0; }
int petiga_cuda_memcpy_d2h(void* dst, const void* src, size_t bytes) { PC_CUDA(cudaMemcpy(dst, src, bytes, cudaMemcpyDeviceToHost)); return 0; }
int petiga_cuda_memset(void* dst, int value, size_t bytes) { PC_CUDA(cudaMemset(dst, value, bytes)); return 0; }
int petiga_cuda_memset_async(petiga_cuda_plan* P, void* dst, int value, size_t bytes) {
  if (!P || (!dst && bytes)) return PETIGA_CUDA_ERR_ARG;
  PC_CUDA(cudaSetDevice(P->device));
  PC_CUDA(cudaMemsetAsync(dst, value, bytes, P->stream));
  return 0;
}
// Pinned host memory on the NUMA node of the current device: the pages are placed by first touch, so the calling thread is moved onto
// the GPU's local CPUs (sysfs local_cpulist of its PCI function) for the allocation and the first touch, then moved back.  With eight
// ranks copying results out at once, buffers that all sit on one socket share one memory controller and one inter-socket link
// (round 1: 10.9 GB/s per GPU at N = 8 against 56.6 GB/s at N = 1).  No sysfs entry (containers, single-socket hosts): plain allocation.
int petiga_cuda_host_alloc(void** ptr, size_t bytes) {
  if (!ptr) return PETIGA_CUDA_ERR_ARG;
  cpu_set_t old_mask, new_mask;
  bool moved = false;
  int dev = 0;
  char bus[32] = {0};
  if (cudaGetDevice(&dev) == cudaSuccess && cudaDeviceGetPCIBusId(bus, sizeof(bus), dev) == cudaSuccess && sched_getaffinity(0, sizeof(old_mask), &old_mask) == 0) {
    for (char* c = bus; *c; c++) *c = (char)tolower(*c);
    const std::string path = std::string("/sys/bus/pci/devices/") + bus + "/local_cpulist";
    if (FILE* f = fopen(path.c_str(), "r")) {
      char line[4096] = {0};
      if (fgets(line, sizeof(line), f)) {
        CPU_ZERO(&new_mask);
        int ncpu = 0;
        for (char* tok = strtok(line, ",\n"); tok; tok = strtok(nullptr, ",\n")) {
          int a = 0, b = 0;
          const int k = sscanf(tok, "%d-%d", &a, &b);
          if (k == 1) b = a;
          if (k >= 1) for (int c = a; c <= b && c < CPU_SETSIZE; c++) if (CPU_ISSET(c, &old_mask)) { CPU_SET(c, &new_mask); ncpu++; }
        }
        if (ncpu > 0 && sched_setaffinity(0, sizeof(new_mask), &new_mask) == 0) moved = true;
      }
      fclose(f);
    }
  } else (void)cudaGetLastError();
  const cudaError_t e = cudaMallocHost(ptr, bytes ? bytes : 1);
  if (e == cudaSuccess && bytes) memset(*ptr, 0, bytes);       // first touch while the thread sits next to the device
  if (moved) sched_setaffinity(0, sizeof(old_mask), &old_mask);
  PC_CUDA(e);
  return 0;
}
int petiga_cuda_host_free(void* ptr) { PC_CUDA(cudaFreeHost(ptr)); return 0; }

int petiga_cuda_plan_exchange_info(petiga_cuda_plan* P, int kind, int* count, int* out, int capacity) {
  if (!P || !count) return PETIGA_CUDA_ERR_ARG;
  const Layout& L = P->L;
  if (kind == 0) {
    *count = (int)L.send.size();
    if (out) for (int i = 0; i < *count && i < capacity; i++) { out[3 * i] = L.send[i].rank; out[3 * i + 1] = L.send[i].first_row; out[3 * i + 2] = L.send[i].nrows; }
  } else {
    *count = (int)L.recv.size();
    if (out) for (int i = 0; i < *count && i < capacity; i++) { out[3 * i] = L.recv[i].rank; out[3 * i + 1] = L.recv[i].rows.empty() ? -1 : L.recv[i].rows[0]; out[3 * i + 2] = (int)L.recv[i].rows.size(); }
  }
  return 0;
}

}  // extern "C"
