// pc_quad3.cuh -- third-generation quadrature kernel: persistent, warp-specialised, FP64 tensor cores, shared-memory scatter.
//
// Same contract as quad_sf_kernel (pc_quad2.cuh) -- the body of the reference's element loop (src/petigaelem.c:375-410,
// 693-1033,1166-1559; src/petigapoint.c:414-492) for 3-D, dof 1, degree 3 with the default 4-point rule, constant-coefficient
// forms on identity or mapped (non-rational) geometry: the headline configuration on the general quadrature path.  What changed,
// each step on a measurement (tools/microbench.cu, profiles/r2_microbench.json; DESIGN.md 3.2b):
//
//  * red.global.add.f64 runs at <= 258 G/s on a B200 (1.09 cycles per lane and SM): the 8.6e9 element-matrix entries of
//    BASELINE cfg 2 cost >= 33 ms of LSU time however fast the arithmetic is.  A CTA therefore walks a whole PENCIL of elements
//    along axis 0 and sums the contributions of consecutive elements in a shared-memory window S[row slot][...] with plain
//    conflict-free LDS/DADD/STS (2.26 T/s); a row slice is flushed with coalesced reductions when no later element of the
//    pencil touches it: 7/16 of the reductions, in runs of 28 contiguous doubles.
//  * mma.sync.m8n8k4.f64 (SASS DMMA) sustains 37.1 TFLOP/s against 34.1 for DFMA, at 1/8 of the issue slots: the three
//    sum-factorisation stages are GEMMs  U1 = PP0 x D',  U2 = U1 x PP1,  K = PP2 x U2  with 16x16 tiles at p = 3; stage A's
//    accumulator fragment is stage B's A operand as it stands (columns <-> contraction index), so only U2 crosses shared memory.
//  * the CTA is split into an ASSEMBLY group (8 warps: stages A-C, window, flush) and a GEOMETRY group (4 warps: 1-D tables by
//    cp.async.bulk (SASS UBLKCP) + mbarrier transaction counts, closure, geometry map and its inverse at the points, D', the
//    element vector) that runs one element ahead through a two-slot ring guarded by full/empty mbarriers (SASS SYNCS); the groups
//    use named barriers (bar.sync 1 / 2), never __syncthreads().
#pragma once
#include "pc_quad2.cuh"

namespace pc {

constexpr int k3AsmThreads = 256, k3Threads = k3AsmThreads + 32;   // 8 assembly warps + 1 producer warp
constexpr int k3Ring = 4;         // ring slots of (PP0 slice, D' block) filled by cp.async.bulk
constexpr int k3U2Q = 388;        // q2 stride of U2 (16 rows of 24 + 4: conflict-free B fragments in stage C)
constexpr int k3MaxPairs = 16;
constexpr int k3SA = 113;         // window S[row slot (4)][a2][a1][e = c0 + 7 (b1 + 4 b2)]: 112 entries in flush (storage) order + 1 pad, so that
constexpr int k3SSlot = 16 * k3SA; //   both the fragment update of stage C and the linear flush walk 16 distinct bank pairs per half-warp
constexpr int k3SSize = 4 * k3SSlot;
constexpr int k3MaxRows = 160;    // axis-0 rows of one pencil segment (tables live in shared memory)
constexpr int k3MaxSeg = 157;     // elements of one pencil segment

struct SF3Params {
  KParams k;
  SFLists l;
  const double* pp[3];            // [e][os*3+ot][a*4+b][q]  (q fastest: A/B fragments are 32 consecutive doubles)
  double* dprime;                 // mapped geometry: D'[local element][pair][64] written by sf3_geom_kernel (swizzled, see d3_index)
  double cconst[k3MaxPairs];      // identity geometry: D'[pair] / JW
  double Cc[16];                  // the form's constant coefficient tensor [NA][NA]
  double fconst[4];               // constant vector coefficient (when !per_qp)
  double C4[16], f4[4];           // the same tensors zero-padded in the canonical physical order [N, d/dx0, d/dx1, d/dx2]
  int c4_n;                       // C4 has entries in the N row / column
  int vslots;                     // bit s: tensor slot s can receive a load term (geometry pre-pass: the other slots are skipped)
  int const_dp;
  int npencils, seglen, nseg;     // work items = npencils * nseg segments of <= seglen elements along axis 0
  int fixsys;                     // slot == SYSTEM with boundary conditions
  int want_mat, want_vec;
};

// position of quadrature point (q0,q1,q2) inside a pair's 64 doubles: q1 is XOR-swizzled with the parity of q2 so that the
// B fragment of stage A (lanes = (q0, q1 in a pair of values, q2 parity)) touches 16 distinct bank pairs per half-warp
__host__ __device__ inline int d3_index(int q0, int q1, int q2) { return q0 + 4 * (q1 ^ (2 * (q2 & 1))) + 16 * q2; }

// plan-level table for this kernel: PP3[e][oo][ab][q]
static __global__ void sf3_pp_kernel(DevAxis ax, double* __restrict__ out) {
  const int per = 9 * 16 * 4;
  const size_t total = (size_t)ax.nel * per;
  for (size_t t = blockIdx.x * (size_t)blockDim.x + threadIdx.x; t < total; t += (size_t)gridDim.x * blockDim.x) {
    const int e = (int)(t / per), r = (int)(t - (size_t)e * per), oo = r / 64, ab = (r / 4) % 16, q = r % 4, a = ab / 4, b = ab % 4;
    const double* v = ax.value + ((size_t)(e * 4 + q) * 4) * 5;
    out[t] = v[a * 5 + oo / 3] * v[b * 5 + oo % 3];
  }
}

__device__ __forceinline__ uint32_t s3_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* b, int count) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(s3_u32(b)), "r"(count)); }
__device__ __forceinline__ void mbar_arrive(uint64_t* b) { asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(s3_u32(b)) : "memory"); }
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* b, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(s3_u32(b)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* b, uint32_t parity, int tag = 0) {
  uint32_t ok = 0;
#ifdef PC_SF3_DEBUG
  long long spins = 0;
#endif
  while (!ok) {
    asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }" : "=r"(ok) : "r"(s3_u32(b)), "r"(parity) : "memory");
#ifdef PC_SF3_DEBUG
    if (++spins > 2000000) { if ((threadIdx.x & 31) == 0) printf("mbar_wait hang: block %d tid %d tag %d parity %u\n", blockIdx.x, threadIdx.x, tag, parity); __trap(); }
#endif
  }
}
__device__ __forceinline__ void mbar_wait_backoff(uint64_t* b, uint32_t parity) {   // the producer's wait: suspend instead of polling
  uint32_t ok = 0;
  while (!ok)   // suspend-time hint (ns): the thread sleeps in hardware until the phase completes or the time is up
    asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3; selp.u32 %0, 1, 0, p; }"
                 : "=r"(ok) : "r"(s3_u32(b)), "r"(parity), "r"(20000u) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* b) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(s3_u32(dst)), "l"(src), "r"(bytes), "r"(s3_u32(b)) : "memory");
}
__device__ __forceinline__ void bar_asm() { asm volatile("bar.sync 1, 256;" ::: "memory"); }
__device__ __forceinline__ void dmma(double& c0, double& c1, double a, double b) {
  asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}

// Dirichlet value / Neumann load of local node (a0,a1,a2) of element ID (dof = 1): BuildFix / AddFixa / AddFlux, petigaelem.c:1166-1283
__device__ __forceinline__ void sf3_node_bc(const KParams& prm, const int ID[3], const int ai[3], int gidx, int& onfix, double& vfix, double& vflux, int pdeg = 3) {
  onfix = 0; vfix = 0.0; vflux = 0.0;
#pragma unroll
  for (int d = 0; d < 3; d++) {
    if (prm.ax[d].periodic) continue;
    for (int s = 0; s < 2; s++) {
      const FixSide& fs = prm.bc[d][s];
      if (!(fs.vcount || fs.lcount)) continue;
      if (ID[d] != (s ? prm.ax[d].nel - 1 : 0)) continue;
      if (ai[d] != (s ? pdeg : 0)) continue;
      for (int k = 0; k < fs.vcount; k++) if (fs.vfield[k] == 0) { onfix = 1; vfix = prm.fixtable ? prm.fixtable[gidx] : fs.vvalue[k]; }
      if (fs.lcount) {
        double A = 1.0;
        for (int e = 0; e < 3; e++) if (e != d) A *= prm.ax[e].detJac[ID[e]] / (double)(pdeg + 1);   // detJac / nen (petigaelem.c:1139)
        if (prm.face_dS[d][s]) {
          const int f0 = (d == 0) ? 1 : 0, f1 = (d == 2) ? 1 : 2;
          A *= prm.face_dS[d][s][(ID[f0] - prm.ax[f0].es) + prm.ax[f0].ew * (ID[f1] - prm.ax[f1].es)];
        } else A *= 4.0;
        for (int k = 0; k < fs.lcount; k++) if (fs.lfield[k] == 0) vflux += fs.lvalue[k] * A;
      }
    }
  }
}
__device__ __forceinline__ bool sf3_elem_on_bc(const KParams& prm, const int ID[3], bool values_only) {
  bool hit = false;
  if (prm.any_bc)
#pragma unroll
    for (int d = 0; d < 3; d++)
      if (!prm.ax[d].periodic) {
        const bool lo = ID[d] == 0, hi = ID[d] == prm.ax[d].nel - 1;
        hit = hit || (lo && (prm.bc[d][0].vcount || (!values_only && prm.bc[d][0].lcount))) || (hi && (prm.bc[d][1].vcount || (!values_only && prm.bc[d][1].lcount)));
      }
  return hit;
}

// ------------------------------------------------------------------------------------------------------------------------
// Geometry pre-pass: one 64-thread CTA per element, many CTAs per SM (latency tolerant).  Writes D'[element][pair][64] for the
// matrix kernel (mapped geometry only) and assembles the element vector (K5-K7, K9 vector part, K10 for vectors).
// Round-2 rewrite: the first version spent 6 300 warp instructions per element (as many as the matrix kernel: 21 of the 56 ms of
// cfg 2g) on index arithmetic and on select chains over the run-time component ranges.  Now every loop has compile-time trip
// counts with thread-constant sub-indices (64 threads = 64 nodes = 64 points), and the form's tensors arrive zero-padded in the
// canonical physical order [N, d/dx0, d/dx1, d/dx2] (sp.C4, sp.f4), so the pull-back is plain 3x3 algebra:
//   D'_GG = JW E C_GG E^T,  D'_NG = JW C_NG E^T,  D'_GN = JW E C_GN,  D'_NN = JW C_NN,   f'_G = JW E f_G,  f'_N = JW f_N
// with E[d][i] = d xi_d / d x_i (petigamapinv.f90.in:28-31).  Tensor slots are [N (if present), xi0, xi1, xi2] by construction
// (build_sf_lists), so slot s is physical index s + 1 - hn.
// ------------------------------------------------------------------------------------------------------------------------
// 4-term dot product of two 32-byte aligned shared-memory quadruples (two LDS.128 each instead of four LDS.64)
__device__ __forceinline__ double dot4_aligned(const double* b, const double* x) {
  const double2 b0 = *reinterpret_cast<const double2*>(b), b1 = *reinterpret_cast<const double2*>(b + 2);
  const double2 x0 = *reinterpret_cast<const double2*>(x), x1 = *reinterpret_cast<const double2*>(x + 2);
  return b0.x * x0.x + b0.y * x0.y + b1.x * x1.x + b1.y * x1.y;
}

__global__ void __launch_bounds__(64) sf3_geom_kernel(const __grid_constant__ SF3Params sp) {
  const KParams& prm = sp.k;
  const SFLists& ls = sp.l;
  __shared__ __align__(16) double gB[96], Xs[192], T1[384], T2[576], Ev[768], Fp[256], Dsh[16 * 64];
  __shared__ double wJ[12], pt[12];
  const int gt = threadIdx.x;
  const int NV = prm.vc1 - prm.vc0, NT = ls.NT;
  const bool mapped = prm.X != nullptr;
  const int hn = ls.tN >= 0 ? 1 : 0;
  const int ID[3] = {(int)blockIdx.x + prm.ax[0].es, (int)blockIdx.y + prm.ax[1].es, (int)blockIdx.z + prm.ax[2].es};
  const size_t elin = blockIdx.x + (size_t)gridDim.x * (blockIdx.y + (size_t)gridDim.y * blockIdx.z);
  {  // Bt[d][o][q][a]: 96 values, thread gt loads entries gt and gt + 64 (d = 0/1 and d = 2)
    const int r = gt & 31, o = r >> 4, q = (r >> 2) & 3, a = r & 3, d0 = gt >> 5;
    gB[gt] = prm.ax[d0].value[((size_t)(ID[d0] * 4 + q) * 4 + a) * 5 + o];
    if (gt < 32) gB[64 + gt] = prm.ax[2].value[((size_t)(ID[2] * 4 + q) * 4 + a) * 5 + o];
  }
  if (gt < 12) {
    const int d = gt >> 2, q = gt & 3;
    wJ[gt] = prm.ax[d].weight[ID[d] * 4 + q] * prm.ax[d].detJac[ID[d]];
    pt[gt] = prm.ax[d].point[ID[d] * 4 + q];
  }
  const int a = gt, ai[3] = {a & 3, (a >> 2) & 3, a >> 4};
  const int gidx = closure_index<3>(prm.ax, ID, ai);
  if (mapped) {
#pragma unroll
    for (int i = 0; i < 3; i++) Xs[i * 64 + a] = prm.X[(size_t)gidx * 3 + i];
  }
  __syncthreads();
  const int q0 = gt & 3, q1 = (gt >> 2) & 3, q2 = gt >> 4;       // this thread's quadrature point (and, as a0 a1 a2, its node)
  if (mapped) {   // X1 = dX/du and X0 at the points by sum factorisation (petigamapgeo.f90.in:28-43)
    {  // T1[i][o0][q0'][a12]:  t = gt + 64 m  ->  i = m >> 1, o0 = m & 1, q0' = gt >> 4, a12 = gt & 15
      const int qq = gt >> 4, a12 = gt & 15;
#pragma unroll
      for (int m = 0; m < 6; m++) {
        const double* b = gB + (m & 1) * 16 + qq * 4;
        const double* x = Xs + (m >> 1) * 64 + a12 * 4;
        T1[gt + 64 * m] = dot4_aligned(b, x);
      }
    }
    __syncthreads();
    {  // T2[i][oc][q0'][q1'][a2]:  t = gt + 64 m  ->  i = m / 3, oc = m % 3 (0 = (1,0), 1 = (0,1), 2 = (0,0)), (q0', q1', a2) from gt
      const int qa = gt >> 4, qb = (gt >> 2) & 3, a2 = gt & 3;
#pragma unroll
      for (int m = 0; m < 9; m++) {
        constexpr int dummy = 0; (void)dummy;
        const int i = m / 3, oc = m % 3, o0 = (oc == 0), o1 = (oc == 1);
        const double* b = gB + 32 + o1 * 16 + qb * 4;
        const double* sx = T1 + i * 128 + o0 * 64 + qa * 16 + a2 * 4;
        T2[gt + 64 * m] = dot4_aligned(b, sx);
      }
    }
    __syncthreads();
    {  // Ev[i][d][q]:  t = gt + 64 m  ->  i = m >> 2, d = m & 3 (3: the point itself), q = gt
#pragma unroll
      for (int m = 0; m < 12; m++) {
        const int i = m >> 2, d = m & 3, oc = (d == 0) ? 0 : (d == 1 ? 1 : 2), o2 = (d == 2);
        const double* b = gB + 64 + o2 * 16 + q2 * 4;
        const double* sx = T2 + i * 192 + oc * 64 + q0 * 16 + q1 * 4;
        Ev[gt + 64 * m] = dot4_aligned(b, sx);
      }
    }
    // (each thread reads back only what it wrote: Ev[.][.][gt]; no barrier)
  }
  {  // one thread per quadrature point: inverse map (petigamapinv.f90.in:28-31), weights, D', vector coefficient
    const int q = gt;
    double E[3][3] = {{1, 0, 0}, {0, 1, 0}, {0, 0, 1}}, x[3] = {pt[q0], pt[4 + q1], pt[8 + q2]};
    double jw = wJ[q0] * wJ[4 + q1] * wJ[8 + q2];                // W = iW jW kW, J = iJ jJ kJ (petiga3d.F90:22-28)
    if (mapped) {
      double X1[3][3];
#pragma unroll
      for (int i = 0; i < 3; i++) {
#pragma unroll
        for (int d = 0; d < 3; d++) X1[i][d] = Ev[i * 256 + d * 64 + q];
        x[i] = Ev[i * 256 + 192 + q];
      }
      const double a00 = X1[0][0], a01 = X1[0][1], a02 = X1[0][2], a10 = X1[1][0], a11 = X1[1][1], a12 = X1[1][2], a20 = X1[2][0], a21 = X1[2][1], a22 = X1[2][2];
      const double det = a00 * (a11 * a22 - a12 * a21) - a01 * (a10 * a22 - a12 * a20) + a02 * (a10 * a21 - a11 * a20);
      const double idet = 1.0 / det;                             // one division instead of nine (each is ~25 instructions)
      E[0][0] = (a11 * a22 - a12 * a21) * idet; E[0][1] = -(a01 * a22 - a02 * a21) * idet; E[0][2] = (a01 * a12 - a02 * a11) * idet;
      E[1][0] = -(a10 * a22 - a12 * a20) * idet; E[1][1] = (a00 * a22 - a02 * a20) * idet; E[1][2] = -(a00 * a12 - a02 * a10) * idet;
      E[2][0] = (a10 * a21 - a11 * a20) * idet; E[2][1] = -(a00 * a21 - a01 * a20) * idet; E[2][2] = (a00 * a11 - a01 * a10) * idet;
      jw *= det;                                                 // detJac *= detX (petigaelem.c:1024-1029)
    }
    if (sp.want_mat && sp.dprime) {
      // D'4 in physical-slot order [N, xi0, xi1, xi2] into this thread's column of Dsh, then the form's pairs out of it
      double Bm[3][3];                                           // B[i][d'] = sum_j C_GG[i][j] E[d'][j]
#pragma unroll
      for (int i = 0; i < 3; i++)
#pragma unroll
        for (int dp = 0; dp < 3; dp++) Bm[i][dp] = sp.C4[(1 + i) * 4 + 1] * E[dp][0] + sp.C4[(1 + i) * 4 + 2] * E[dp][1] + sp.C4[(1 + i) * 4 + 3] * E[dp][2];
#pragma unroll
      for (int d = 0; d < 3; d++)
#pragma unroll
        for (int dp = 0; dp < 3; dp++) Dsh[((1 + d) * 4 + 1 + dp) * 64 + q] = jw * (E[d][0] * Bm[0][dp] + E[d][1] * Bm[1][dp] + E[d][2] * Bm[2][dp]);
      if (sp.c4_n) {                                             // the form couples N (mass / reaction terms)
        Dsh[q] = jw * sp.C4[0];
#pragma unroll
        for (int d = 0; d < 3; d++) {
          Dsh[(1 + d) * 64 + q] = jw * (sp.C4[1] * E[d][0] + sp.C4[2] * E[d][1] + sp.C4[3] * E[d][2]);                  // D'[N][xi_d]
          Dsh[((1 + d) * 4) * 64 + q] = jw * (E[d][0] * sp.C4[4] + E[d][1] * sp.C4[8] + E[d][2] * sp.C4[12]);           // D'[xi_d][N]
        }
      }
      double* D = sp.dprime + elin * ls.npairs * 64 + d3_index(q0, q1, q2);
      const int sh = 1 - hn;
      for (int pr = 0; pr < ls.npairs; pr++) D[(size_t)pr * 64] = Dsh[((ls.pair_s[pr] + sh) * 4 + ls.pair_t[pr] + sh) * 64 + q];
    }
    if (sp.want_vec && NV > 0) {
      double f4[4] = {sp.f4[0], sp.f4[1], sp.f4[2], sp.f4[3]};
      if (prm.per_qp) {
        QPoint qp;
        qp.atboundary = 0;
        qp.x[0] = x[0]; qp.x[1] = x[1]; qp.x[2] = x[2];
        double fv[4] = {0.0, 0.0, 0.0, 0.0};
        form_coefficients<3, 1>(prm.form, prm.slot, prm.prm, prm.shift, prm.t, qp, 0, NV, nullptr, fv);
#pragma unroll
        for (int ca = 0; ca < 4; ca++) {
          f4[ca] = 0.0;
#pragma unroll
          for (int al = 0; al < 4; al++) if (al < NV && prm.vc0 + al == ca) f4[ca] = fv[al];
        }
      }
      // f'[slot][q]: N slot (if present) first, then the three parametric gradients
      if (hn) Fp[q] = jw * f4[0];
#pragma unroll
      for (int d = 0; d < 3; d++)
        if (hn + d < NT) Fp[(hn + d) * 64 + q] = jw * (E[d][0] * f4[1] + E[d][1] * f4[2] + E[d][2] * f4[3]);
    }
  }
  if (!sp.want_vec) return;
  // ---- element vector by the transposed sum factorisation, fix-up, scatter ----
  double F = 0.0;
  if (NV > 0) {
    __syncthreads();
    double* R1 = T1;                                           // [s][q2][q1][a0]
    double* R2 = T2;                                           // [s][q2][a1][a0]
    {
      const int q12 = gt >> 2, a0 = gt & 3;                    // t = gt + 64 s
      for (int sl = 0; sl < NT; sl++) {
        if (!((sp.vslots >> sl) & 1)) continue;                  // slots the load never feeds (Poisson: only N) are skipped in all three stages
        const double* f = Fp + sl * 64 + q12 * 4;
        const double* b = gB + ls.torder[sl][0] * 16 + a0;
        R1[gt + 64 * sl] = b[0] * f[0] + b[4] * f[1] + b[8] * f[2] + b[12] * f[3];
      }
    }
    __syncthreads();
    {
      const int qq2 = gt >> 4, a1 = (gt >> 2) & 3, a0 = gt & 3;
      for (int sl = 0; sl < NT; sl++) {
        if (!((sp.vslots >> sl) & 1)) continue;
        const double* b = gB + 32 + ls.torder[sl][1] * 16 + a1;
        const double* xx = R1 + sl * 64 + qq2 * 16 + a0;
        R2[gt + 64 * sl] = b[0] * xx[0] + b[4] * xx[4] + b[8] * xx[8] + b[12] * xx[12];
      }
    }
    __syncthreads();
    const int a2 = a >> 4, a01 = a & 15;
    for (int sl = 0; sl < NT; sl++) {
      if (!((sp.vslots >> sl) & 1)) continue;
      const double* b = gB + 64 + ls.torder[sl][2] * 16 + a2;
      const double* xx = R2 + sl * 64 + a01;
      F += b[0] * xx[0] + b[4] * xx[16] + b[8] * xx[32] + b[12] * xx[48];
    }
  }
  if (prm.slot == PETIGA_SLOT_SYSTEM && sf3_elem_on_bc(prm, ID, false)) {          // FixSystem vector part (petigaelem.c:1365-1387)
    int onfix; double vfix, vflux;
    sf3_node_bc(prm, ID, ai, gidx, onfix, vfix, vflux);
    F += vflux;
    if (onfix) F = vfix;
  }
  if (F != 0.0) atomicAdd(&prm.rhs[prm.localrow[gidx]], F);
}

struct SF3Smem {   // offsets in doubles
  int S, U2, PP1, PP2, ring, rowoff, seg0, W0, wj0, offT, PT, fix, bars, total, slot;
  __host__ __device__ SF3Smem(int npairs, int mapped) {
    int o = 0;
    S = o; o += k3SSize;
    U2 = o; o += 4 * 4 * k3U2Q;
    PP1 = o; o += 576; PP2 = o; o += 576;
    slot = 576 + (mapped ? npairs * 64 : 0);           // one ring slot: PP0 slice, then D' of the element
    ring = o; o += k3Ring * slot;
    rowoff = o; o += k3MaxRows * 16;                   // int64 per (axis-0 row, a1, a2)
    seg0 = o; o += k3MaxRows * 8 / 2;                  // uint32 [row][8]
    W0 = o; o += k3MaxRows / 2;                        // int32
    wj0 = o; o += k3MaxSeg * 4 + 4;                    // axis-0 weight * detJac per (element, q0)
    offT = o; o += (k3MaxSeg + 3) / 2 + 1;             // int32: first row of every element, relative to the segment
    PT = o; o += 128;
    fix = o; o += 64 + 32 + 32;                        // fixval[64], fixflag int[64], rowlr int[64] of a boundary element
    bars = o; o += 2 * k3Ring;
    total = o;
  }
};

__global__ void __launch_bounds__(k3Threads, 1) quad_sf3_kernel(const __grid_constant__ SF3Params sp) {
  const KParams& prm = sp.k;
  const SFLists& ls = sp.l;
  extern __shared__ __align__(128) double sm3[];
  const bool mapped = prm.X != nullptr;
  const SF3Smem lay(ls.npairs, mapped ? 1 : 0);
  double *S = sm3 + lay.S, *U2 = sm3 + lay.U2, *PP1 = sm3 + lay.PP1, *PP2 = sm3 + lay.PP2, *Ring = sm3 + lay.ring;
  int64_t* rowoffT = reinterpret_cast<int64_t*>(sm3 + lay.rowoff);
  uint32_t* seg0T = reinterpret_cast<uint32_t*>(sm3 + lay.seg0);
  int* W0T = reinterpret_cast<int*>(sm3 + lay.W0);
  double* wj0T = sm3 + lay.wj0;
  int* offT = reinterpret_cast<int*>(sm3 + lay.offT);
  uint32_t* PT = reinterpret_cast<uint32_t*>(sm3 + lay.PT);
  double* fixval = sm3 + lay.fix;
  int* fixflag = reinterpret_cast<int*>(sm3 + lay.fix + 64);
  int* rowlr = fixflag + 64;
  uint64_t* full = reinterpret_cast<uint64_t*>(sm3 + lay.bars);
  uint64_t* empty = full + k3Ring;
  const int tid = threadIdx.x;
  const int ew0 = prm.ax[0].ew, ew1 = prm.ax[1].ew;
  const int nwork = sp.npencils * sp.nseg;
  const uint32_t slot_bytes = (uint32_t)lay.slot * 8;

  if (tid == 0) {
    for (int k = 0; k < k3Ring; k++) { mbar_init(&full[k], 1); mbar_init(&empty[k], k3AsmThreads / 32); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  for (int t = tid; t < k3SSize; t += k3Threads) S[t] = 0.0;
  __syncthreads();

  if (tid >= k3AsmThreads) {
    // ===================== PRODUCER WARP: cp.async.bulk of (PP0 slice, D') per element into the ring =====================
    if (tid == k3AsmThreads) {
      uint32_t it = 0;
      for (int w = blockIdx.x; w < nwork; w += gridDim.x) {
        const int pen = w / sp.nseg, seg = w - pen * sp.nseg;
        const int l1 = pen % ew1, l2 = pen / ew1;
        const int le0 = seg * sp.seglen, le1 = min(ew0, le0 + sp.seglen);
        for (int le = le0; le < le1; le++, it++) {
          const int slot = it % k3Ring;
          mbar_wait_backoff(&empty[slot], ((it / k3Ring) & 1) ^ 1);
          double* dst = Ring + (size_t)slot * lay.slot;
          mbar_arrive_expect_tx(&full[slot], slot_bytes);
          bulk_g2s(dst, sp.pp[0] + (size_t)(prm.ax[0].es + le) * 576, 576 * 8, &full[slot]);
          if (mapped) {
            const size_t el = (size_t)le + (size_t)ew0 * (l1 + (size_t)ew1 * l2);
            bulk_g2s(dst + 576, sp.dprime + el * ls.npairs * 64, (uint32_t)ls.npairs * 512, &full[slot]);
          }
        }
      }
    }
    return;
  }

  // =========================================== ASSEMBLY GROUP ===========================================
  const int lane = tid & 31, warp = tid >> 5, r = lane >> 2, c = lane & 3;
  int fc0[4], fbb[4];                                   // flush: a lane owns entries e = lane + 32 k of a row's 112 (c0 fastest, then b1, b2)
#pragma unroll
  for (int k = 0; k < 4; k++) { const int e = lane + 32 * k; fc0[k] = e % 7; fbb[k] = e / 7; }
  const int q1l = r >> 1, parl = r & 1;                 // this lane's (q1, q2 parity) as column of stage A
  const int dfrag = c + 4 * (q1l ^ (2 * parl)) + 16 * parl;   // + 32 b: d3_index(c, q1l, 2 b + parl)
  uint32_t it = 0;
  for (int w = blockIdx.x; w < nwork; w += gridDim.x) {
    const int pen = w / sp.nseg, seg = w - pen * sp.nseg;
    const int e1 = prm.ax[1].es + pen % ew1, e2 = prm.ax[2].es + pen / ew1;
    const int le0 = seg * sp.seglen, le1 = min(ew0, le0 + sp.seglen), nel = le1 - le0;
    const int G1 = prm.ax[1].offset[e1] - prm.ax[1].gs, G2 = prm.ax[2].offset[e2] - prm.ax[2].gs;
    const int off_first = prm.ax[0].offset[prm.ax[0].es + le0];
    const int Gf = off_first - prm.ax[0].gs;                            // ghost coordinate of the segment's first row
    const int nrows = prm.ax[0].offset[prm.ax[0].es + le1 - 1] - off_first + 4;
    bar_asm();                                                         // previous work item's readers of the tables are done
    {
      const double* g1p = sp.pp[1] + (size_t)e1 * 576;
      const double* g2p = sp.pp[2] + (size_t)e2 * 576;
      for (int t = tid; t < 576; t += k3AsmThreads) { PP1[t] = g1p[t]; PP2[t] = g2p[t]; }
      {  // PT[(a1,a2)][(b1,b2)]: pos = P1*W0 + P2*Bi + P3*Si + Li
        const int a12 = tid >> 4, bb = tid & 15, a1 = a12 & 3, a2 = a12 >> 2, b1 = bb & 3, b2 = bb >> 2;
        const int g1 = G1 + a1, g2 = G2 + a2;
        const uint32_t s1 = prm.ax[1].seg[g1 * kMaxW + b1 - a1 + prm.ax[1].lo[g1]], s2 = prm.ax[2].seg[g2 * kMaxW + b2 - a2 + prm.ax[2].lo[g2]];
        const int Bj = s1 & 255, Sj = (s1 >> 8) & 255, Lj = (s1 >> 16) & 255, Bk = s2 & 255, Sk = (s2 >> 8) & 255, Lk = (s2 >> 16) & 255;
        const int W1 = prm.ax[1].W[g1];
        PT[tid] = (uint32_t)(Bk * W1 + Sk * Bj) | ((uint32_t)(Sk * Sj) << 16) | ((uint32_t)(Lk * Sj + Lj) << 24);
      }
      // the rows of this pencil segment: value offsets, axis-0 position bytes and widths -- no global loads inside the element loop
      for (int t = tid; t < nrows * 16; t += k3AsmThreads) {
        const int i0 = t >> 4, a12 = t & 15, a1 = a12 & 3, a2 = a12 >> 2;
        const int gidx = (Gf + i0) + prm.ax[0].gw * ((G1 + a1) + prm.ax[1].gw * (G2 + a2));
        const int lr = prm.localrow[gidx];
        int64_t base = prm.rowbase[lr];
        if (lr >= prm.nown) base = (base - prm.nnz_own) | ((int64_t)1 << 62);
        rowoffT[t] = base;
      }
      for (int t = tid; t < nrows * 8; t += k3AsmThreads) {
        const int i0 = t >> 3, c0 = t & 7, g = Gf + i0;
        const int W = prm.ax[0].W[g], cc = c0 - 3 + prm.ax[0].lo[g];
        if (c0 < 7) seg0T[t] = (cc >= 0 && cc < W) ? prm.ax[0].seg[g * kMaxW + cc] : 0xFFFFFFFFu;
        else seg0T[t] = (uint32_t)prm.ax[0].simple[g];                  // slot 7: this row's columns are in storage order along axis 0
        if (c0 == 0) W0T[i0] = W;
      }
      for (int t = tid; t < nel * 4; t += k3AsmThreads) {
        const int e0 = prm.ax[0].es + le0 + (t >> 2), q = t & 3;
        wj0T[t] = prm.ax[0].weight[e0 * 4 + q] * prm.ax[0].detJac[e0];
      }
      for (int t = tid; t <= nel; t += k3AsmThreads)
        offT[t] = (t < nel) ? prm.ax[0].offset[prm.ax[0].es + le0 + t] - off_first : nrows;       // sentinel: everything is complete at the end
    }
    // does this pencil touch a Dirichlet face of axis 1 or 2?  (axis 0: first / last element of the mesh)
    bool pen_fix = false, lo0_fix = false, hi0_fix = false;
    if (sp.fixsys) {
      if (!prm.ax[1].periodic) pen_fix = pen_fix || (e1 == 0 && prm.bc[1][0].vcount) || (e1 == prm.ax[1].nel - 1 && prm.bc[1][1].vcount);
      if (!prm.ax[2].periodic) pen_fix = pen_fix || (e2 == 0 && prm.bc[2][0].vcount) || (e2 == prm.ax[2].nel - 1 && prm.bc[2][1].vcount);
      if (!prm.ax[0].periodic) { lo0_fix = prm.bc[0][0].vcount > 0; hi0_fix = prm.bc[0][1].vcount > 0; }
    }
    // identity geometry: D'[pair][q] = cconst[pair] * wJ0[q0] * wJ1[q1] * wJ2[q2]; this lane's q1 and its two q2 values are fixed
    double wq12[2] = {0, 0};
    if (!mapped) {
      const double w1 = prm.ax[1].weight[e1 * 4 + q1l] * prm.ax[1].detJac[e1];
#pragma unroll
      for (int b = 0; b < 2; b++) wq12[b] = w1 * prm.ax[2].weight[e2 * 4 + 2 * b + parl] * prm.ax[2].detJac[e2];
    }
    bar_asm();
    // flush tables of this lane for the whole work item: entry k of row rr of this warp -> window offset, position coefficients
    int fso[2][4], fP1[2][4], fP23[2][4], fP13[2][4];
#pragma unroll
    for (int rr = 0; rr < 2; rr++) {
      const int a12 = 2 * warp + rr, a1 = a12 & 3, a2 = a12 >> 2;
#pragma unroll
      for (int k = 0; k < 4; k++) {
        const int c0 = fc0[k], bb = fbb[k] & 15;
        const uint32_t ptv = PT[a12 * 16 + bb];
        fso[rr][k] = (a2 * 4 + a1) * k3SA + lane + 32 * k;
        fP1[rr][k] = (int)(ptv & 0xFFFF);
        fP23[rr][k] = (int)(ptv >> 16);
        fP13[rr][k] = (int)(ptv & 0xFFFF) + (int)(ptv >> 24);          // storage-order rows: pos = (P1 + P3) W0 + c0 - c0first
      }
    }
    for (int le = 0; le < nel; le++, it++) {
      const int slot = it % k3Ring;
      const double* P0 = Ring + (size_t)slot * lay.slot;
      const double* D = P0 + 576;
      const int i0 = offT[le], nflush = min(4, offT[le + 1] - i0);       // rows [i0, i0 + nflush) are complete after this element
      const int IDs[3] = {prm.ax[0].es + le0 + le, e1, e2};
      const bool elem_fix = pen_fix || (lo0_fix && IDs[0] == 0) || (hi0_fix && IDs[0] == prm.ax[0].nel - 1);
      if (elem_fix && tid < 64) {                                        // Dirichlet data of a boundary element (single buffer: see the barriers)
        const int ai[3] = {tid & 3, (tid >> 2) & 3, tid >> 4};
        const int gidx = (Gf + i0 + ai[0]) + prm.ax[0].gw * ((G1 + ai[1]) + prm.ax[1].gw * (G2 + ai[2]));
        int onfix; double vfix, vflux;
        sf3_node_bc(prm, IDs, ai, gidx, onfix, vfix, vflux);
        fixflag[tid] = onfix; fixval[tid] = vfix; rowlr[tid] = prm.localrow[gidx];
      }
      const double w0q = mapped ? 0.0 : wj0T[le * 4 + c];
      mbar_wait(&full[slot], (it / k3Ring) & 1);                         // the PP0 slice (and D') of this element have landed
      // ---- stages A + B: a warp owns the combos (g2, q2) = combo, combo + 8, ...; stage A's accumulators feed stage B ----
      for (int combo = warp; combo < ls.ng2 * 4; combo += 8) {
        const int g2 = combo >> 2, q2 = combo & 3, b = q2 >> 1, x = q2 & 1;
        const double wq = w0q * wq12[b];
        double cB[2][2][2] = {{{0, 0}, {0, 0}}, {{0, 0}, {0, 0}}};   // [mt][nt][reg]
        for (int g1 = ls.g2_first[g2]; g1 < ls.g2_first[g2 + 1]; g1++) {
          double cA[2][2] = {{0, 0}, {0, 0}};                        // [mt][reg]: U1[ab0 = r + 8 mt][q1 = c][q2 = 2b + reg]
          for (int pr = ls.g1_first[g1]; pr < ls.g1_first[g1 + 1]; pr++) {
            const double bf = mapped ? D[pr * 64 + dfrag + 32 * b] : sp.cconst[pr] * wq;
            const double* pa = P0 + ls.pair_oo0[pr] * 64 + lane;
            dmma(cA[0][0], cA[0][1], pa[0], bf);
            dmma(cA[1][0], cA[1][1], pa[32], bf);
          }
          const double* pb = PP1 + ls.g1_oo1[g1] * 64 + lane;
          const double b0 = pb[0], b1 = pb[32];
          const double ax0 = x ? cA[0][1] : cA[0][0], ax1 = x ? cA[1][1] : cA[1][0];   // (a select, not a dynamic index: no local memory)
          dmma(cB[0][0][0], cB[0][0][1], ax0, b0);
          dmma(cB[0][1][0], cB[0][1][1], ax0, b1);
          dmma(cB[1][0][0], cB[1][0][1], ax1, b0);
          dmma(cB[1][1][0], cB[1][1][1], ax1, b1);
        }
        double* u = U2 + (g2 * 4 + q2) * k3U2Q + r * 24 + 2 * c;     // U2[g2][q2][ab0 * 24 + ab1]
#pragma unroll
        for (int mt = 0; mt < 2; mt++)
#pragma unroll
          for (int nt = 0; nt < 2; nt++)
            *reinterpret_cast<double2*>(u + mt * 8 * 24 + nt * 8) = make_double2(cB[mt][nt][0], cB[mt][nt][1]);
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&empty[slot]);                        // this warp no longer reads the ring slot
      bar_asm();
      {
        // ---- stage C: K[ab2][ab1][ab0] for ab0 in {2 warp, 2 warp + 1}; k index = q2 ----
        double cC[2][2][2][2];                                         // [h][nt][mt][reg]
#pragma unroll
        for (int h = 0; h < 2; h++)
#pragma unroll
          for (int nt = 0; nt < 2; nt++)
#pragma unroll
            for (int mt = 0; mt < 2; mt++) cC[h][nt][mt][0] = cC[h][nt][mt][1] = 0.0;
        for (int g2 = 0; g2 < ls.ng2; g2++) {
          const double* pa = PP2 + ls.g2_oo2[g2] * 64 + lane;
          const double a0f = pa[0], a1f = pa[32];
          const double* ub = U2 + (g2 * 4 + c) * k3U2Q + (2 * warp) * 24 + r;
#pragma unroll
          for (int h = 0; h < 2; h++)
#pragma unroll
            for (int nt = 0; nt < 2; nt++) {
              const double bf = ub[h * 24 + nt * 8];
              dmma(cC[h][nt][0][0], cC[h][nt][0][1], a0f, bf);
              dmma(cC[h][nt][1][0], cC[h][nt][1][1], a1f, bf);
            }
        }
        // ---- Dirichlet fix-up on the fragments (petigaelem.c:1360-1389), then the shared-memory window ----
        const int a0 = warp >> 1;
        double* sbase = S + ((i0 + a0) & 3) * k3SSlot + ((r >> 2) * 4 + (c >> 1)) * k3SA + (2 * (c & 1) + 4 * (r & 3)) * 7;
        if (!elem_fix) {
#pragma unroll
          for (int h = 0; h < 2; h++) {
            const int c0 = 2 * (warp & 1) + h - a0 + 3;
#pragma unroll
            for (int nt = 0; nt < 2; nt++)
#pragma unroll
              for (int mt = 0; mt < 2; mt++) {
                double* sp0 = sbase + (8 * mt + 2 * nt) * k3SA + c0;
                sp0[0] += cC[h][nt][mt][0];
                sp0[7] += cC[h][nt][mt][1];
              }
          }
        } else {
#pragma unroll
          for (int h = 0; h < 2; h++) {
            const int b0 = 2 * (warp & 1) + h, c0 = b0 - a0 + 3;
#pragma unroll
            for (int nt = 0; nt < 2; nt++)
#pragma unroll
              for (int mt = 0; mt < 2; mt++) {
                const int a2 = 2 * mt + (r >> 2), b2 = r & 3, a1 = 2 * nt + (c >> 1);
                double* sp0 = sbase + (8 * mt + 2 * nt) * k3SA + c0;
#pragma unroll
                for (int x = 0; x < 2; x++) {
                  double v = cC[h][nt][mt][x];
                  const int b1 = 2 * (c & 1) + x, ra = a0 + 4 * a1 + 16 * a2, cb = b0 + 4 * b1 + 16 * b2;
                  const bool fr = fixflag[ra], fcx = fixflag[cb];
                  if (fr || fcx) {
                    if (fcx && !fr) atomicAdd(&prm.rhs[rowlr[ra]], -v * fixval[cb]);
                    v = (ra == cb) ? 1.0 : 0.0;
                  }
                  sp0[7 * x] += v;
                }
              }
          }
        }
      }
      bar_asm();
      // ---- flush the row slots no later element of the segment touches: coalesced red.global.add.f64 ----
      for (int f = 0; f < nflush; f++) {
        const int row = i0 + f, W0 = W0T[row];
        double* srow = S + (row & 3) * k3SSlot;
        const uint32_t sfirst = seg0T[row * 8 + 3];                     // the diagonal column always exists
        // axis 0 in storage order: every existing column c0 has (Bi, Si, Li) = (0, W0, c0 - c0first), so
        // pos = P1 W0 + P2 Bi + P3 Si + Li = (P1 + P3) W0 + c0 - c0first whatever the owners along axes 1 and 2
        const int c0first = 3 - (int)((sfirst >> 16) & 255);
        const bool row_simple = (seg0T[row * 8 + 7] == 1u);            // flag written with the tables
#pragma unroll
        for (int rr = 0; rr < 2; rr++) {
          const int64_t ro = rowoffT[row * 16 + 2 * warp + rr];
          double* dst = ((ro >> 62) & 1) ? prm.ghost_values + (ro & (((int64_t)1 << 62) - 1)) : prm.values + ro;
          if (row_simple) {
            double* dstc = dst - c0first;
            double vv[4];
#pragma unroll
            for (int k = 0; k < 4; k++) vv[k] = (k == 3 && lane >= 16) ? 0.0 : srow[fso[rr][k]];
#pragma unroll
            for (int k = 0; k < 4; k++)
              if (vv[k] != 0.0) { atomicAdd(dstc + (fP13[rr][k] * W0 + fc0[k]), vv[k]); srow[fso[rr][k]] = 0.0; }
          } else {
#pragma unroll
            for (int k = 0; k < 4; k++) {
              if (k == 3 && lane >= 16) break;
              double* sp0 = srow + fso[rr][k];
              const double v = *sp0;
              if (v != 0.0) {
                const uint32_t s0 = seg0T[row * 8 + fc0[k]];
                const int pos = fP1[rr][k] * W0 + (fP23[rr][k] & 255) * (int)(s0 & 255) + (fP23[rr][k] >> 8) * (int)((s0 >> 8) & 255) + (int)((s0 >> 16) & 255);
                atomicAdd(dst + pos, v);
                *sp0 = 0.0;
              }
            }
          }
        }
      }
    }
  }
}

}  // namespace pc
