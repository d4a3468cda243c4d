// pc_quad3.cu -- launcher of the third-generation quadrature kernel (pc_quad3.cuh).
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "pc_plan.h"
#include "pc_quad3r.cuh"
#include "pc_quadv.cuh"

namespace pc {

// tensor slots the load vector can feed: N when the form has a value term, the three gradients when it has a gradient term
static int vector_slots(const KParams& base, const SFLists& l, const double* f4) {
  const int NV = base.vc1 - base.vc0;
  const bool per_qp = base.per_qp != 0;
  const bool fN = base.vc0 == 0 && NV > 0 && (per_qp || f4[0] != 0.0);
  bool fG = false;
  for (int ca = 1; ca < 4; ca++) if (ca >= base.vc0 && ca < base.vc1 && (per_qp || f4[ca] != 0.0)) fG = true;
  int m = 0;
  if (fN && l.tN >= 0) m |= 1 << l.tN;
  if (fG) for (int d = 0; d < 3; d++) if (l.tG[d] >= 0) m |= 1 << l.tG[d];
  return m;
}

// vector-only assembly (pc_quadv.cuh): IGAComputeVector, or the load vector of a system whose matrix the separable path has written
int launch_quadrature_vec3(petiga_cuda_plan* Pl, const KParams& base) {
  const int dim = base.dim, dof = base.dof;
  auto nope = [](const char* why) { set_error(std::string("quad_vec3: ") + why); return PETIGA_CUDA_ERR_SUP; };
  if (dim != 3 || dof != 1) return nope("3-D, one dof per node only");
  const int p = base.ax[0].p;
  if (p < 2 || p > 4) return nope("degree 2..4 only");
  for (int d = 0; d < 3; d++) if (base.ax[d].p != p || base.ax[d].nqp != p + 1) return nope("one degree on all axes with the default rule only");
  if (base.Wt) return nope("rational geometry");
  if (base.mc1 != base.mc0) return nope("vector-only");
  if (base.slot != PETIGA_SLOT_VECTOR && !(base.slot == PETIGA_SLOT_SYSTEM && !base.any_bc)) return nope("IGAComputeVector or an unconstrained system only");
  FormInfo fi = form_info(base.form, base.slot, dim, dof);
  if (!fi.valid || fi.order > 1 || fi.needs_state || base.U) return nope("first-order forms without state only");
  const int NV = base.vc1 - base.vc0;
  if (NV <= 0 || NV > 4) return nope("components");
  SF3Params sp;
  memset(&sp, 0, sizeof(sp));
  sp.k = base;
  std::vector<double> fv((size_t)NV, 0.0);
  {
    QPoint q;
    memset(&q, 0, sizeof(q));
    form_coefficients<3, 1>(base.form, base.slot, base.prm, base.shift, base.t, q, 0, NV, nullptr, fv.data());
  }
  for (int k = 0; k < NV; k++) sp.fconst[k] = fv[k];
  std::vector<char> cpat(1, 0);
  if (build_sf_lists(base, fi, base.X != nullptr, false, false, false, cpat, 0, sp.l)) return nope("component lists");
  if (sp.l.NT > 4) return nope("too many tensor components");
  for (int t = 0; t < sp.l.NT; t++) for (int d = 0; d < 3; d++) if (sp.l.torder[t][d] > 1) return nope("second derivatives");
  for (int al = 0; al < NV; al++) if (base.vc0 + al < 4) sp.f4[base.vc0 + al] = fv[al];
  sp.vslots = vector_slots(base, sp.l, sp.f4);
  sp.want_vec = 1;
  if (base.nelem <= 0) return 0;
  const int n3 = (p + 1) * (p + 1) * (p + 1), threads = (n3 + 31) / 32 * 32;
  if (base.ax[1].ew > 65535 || base.ax[2].ew > 65535) return nope("element box too large for a 3-D grid");
  const dim3 grid3((unsigned)base.ax[0].ew, (unsigned)base.ax[1].ew, (unsigned)base.ax[2].ew);
#define VK(P_) { if (base.X) quad_vec3_kernel<P_, true><<<grid3, threads, 0, Pl->stream>>>(sp); else quad_vec3_kernel<P_, false><<<grid3, threads, 0, Pl->stream>>>(sp); }
  if (p == 2) VK(2) else if (p == 3) VK(3) else VK(4)
#undef VK
  PC_CUDA(cudaGetLastError());
  Pl->launches++;
  const double n4 = (double)(p + 1) * (p + 1) * (p + 1) * (p + 1);
  Pl->last_flops = (double)base.nelem * ((base.X ? 2.0 * n4 * (6 + 9 + 12) : 0.0) + 2.0 * n4 * 3 * sp.l.NT + 60.0 * n3);
  return 0;
}

int launch_quadrature_sf3(petiga_cuda_plan* Pl, const KParams& base) {
  const int dim = base.dim, dof = base.dof;
  auto nope = [](const char* why) { set_error(std::string("quad_sf3: ") + why); return PETIGA_CUDA_ERR_SUP; };
  if (dim != 3 || dof != 1) return nope("3-D, one dof per node only");
  for (int d = 0; d < 3; d++) if (base.ax[d].p != 3 || base.ax[d].nqp != 4) return nope("degree 3 with the default 4-point rule only");
  if (base.Wt) return nope("rational geometry runs the second-generation kernel");
  if (base.slot != PETIGA_SLOT_VECTOR && base.slot != PETIGA_SLOT_MATRIX && base.slot != PETIGA_SLOT_SYSTEM) return nope("linear drivers only");
  FormInfo fi = form_info(base.form, base.slot, dim, dof);
  if (!fi.valid || !fi.mat_const || fi.order > 1 || fi.needs_state || base.U) return nope("constant-coefficient first-order forms only");
  const bool mapped = base.X != nullptr;
  SF3Params sp;
  memset(&sp, 0, sizeof(sp));
  sp.k = base;
  const int NA = base.mc1 - base.mc0, NV = base.vc1 - base.vc0;
  if (NA > 4 || NV > 4) return nope("too many components");
  // the form's constant coefficient tensor and vector (evaluated once on the host at a dummy point)
  std::vector<double> C((size_t)std::max(NA * NA, 1), 0.0), fv((size_t)std::max(NV, 1), 0.0);
  {
    QPoint q;
    memset(&q, 0, sizeof(q));
    form_coefficients<3, 1>(base.form, base.slot, base.prm, base.shift, base.t, q, NA, NV, NA ? C.data() : nullptr, NV ? fv.data() : nullptr);
  }
  std::vector<char> cpat((size_t)std::max(NA * NA, 1), 0);
  for (int k = 0; k < NA * NA; k++) { cpat[k] = C[k] != 0.0; sp.Cc[k] = C[k]; }
  for (int k = 0; k < NV; k++) sp.fconst[k] = fv[k];
  for (int al = 0; al < NA; al++)
    for (int be = 0; be < NA; be++) {
      const int ca = base.mc0 + al, cb = base.mc0 + be;
      if (ca < 4 && cb < 4) { sp.C4[ca * 4 + cb] = C[(size_t)al * NA + be]; if ((ca == 0 || cb == 0) && C[(size_t)al * NA + be] != 0.0) sp.c4_n = 1; }
    }
  for (int al = 0; al < NV; al++) if (base.vc0 + al < 4) sp.f4[base.vc0 + al] = fv[al];
  int rc = build_sf_lists(base, fi, mapped, false, false, false, cpat, NA > 0 ? 1 : 0, sp.l);
  if (rc) return nope("component lists");
  if (sp.l.NT > 4 || sp.l.npairs > k3MaxPairs || sp.l.ng2 > 4) return nope("too many tensor components");
  sp.vslots = vector_slots(base, sp.l, sp.f4);
  // per-axis pair-product tables in the fragment layout, once per plan (into a local buffer, kept once the build has been launched)
  for (int d = 0; d < 3; d++) {
    if (!Pl->d_ax[d].sf3pp) {
      const size_t n = (size_t)base.ax[d].nel * 576;
      DevBuf<double> pp;
      if ((rc = pp.reserve(n))) return rc;
      sf3_pp_kernel<<<(int)std::min<size_t>((n + 255) / 256, 4096), 256, 0, Pl->stream>>>(base.ax[d], pp.get());
      PC_CUDA(cudaGetLastError());
      Pl->launches++;
      Pl->d_ax[d].sf3pp = std::move(pp);
    }
    sp.pp[d] = Pl->d_ax[d].sf3pp.get();
  }
  sp.const_dp = 0;
  if (!mapped && NA > 0) {   // identity geometry: D'[pair] = JW * C[phys(s)][phys(t)]
    sp.const_dp = 1;
    auto phys_of = [&](int t) -> int {
      if (t == sp.l.tN) return 0;
      for (int d = 0; d < 3; d++) if (t == sp.l.tG[d]) return 1 + d;
      return 4;
    };
    for (int pr = 0; pr < sp.l.npairs; pr++) {
      const int al = phys_of(sp.l.pair_s[pr]) - base.mc0, be = phys_of(sp.l.pair_t[pr]) - base.mc0;
      sp.cconst[pr] = (al >= 0 && al < NA && be >= 0 && be < NA) ? C[(size_t)al * NA + be] : 0.0;
    }
  }
  sp.npencils = base.ax[1].ew * base.ax[2].ew;
  sp.fixsys = (base.slot == PETIGA_SLOT_SYSTEM && base.any_bc) ? 1 : 0;
  sp.want_mat = (NA > 0 && slot_has_mat(base.slot)) ? 1 : 0;
  sp.want_vec = slot_has_vec(base.slot) ? 1 : 0;
  bool smooth0 = false;
  {  // pencil segments: the axis-0 rows of a segment must fit the shared-memory tables
    const AxisLayout& a0 = Pl->L.ax[0];
    // rows advance by (offset[e+1] - offset[e]) per element: 1 on a maximally smooth axis, at most p + 1 otherwise
    const int maxstep = (a0.nnp == a0.nel + a0.p || (a0.periodic && a0.nnp == a0.nel)) ? 1 : a0.p + 1;
    smooth0 = (maxstep == 1);
    sp.seglen = std::max(1, std::min(k3MaxSeg, (k3MaxRows - 4) / maxstep + 1));
    sp.nseg = (a0.ew + sp.seglen - 1) / sp.seglen;
  }
  if (base.nelem <= 0) return 0;
  if (mapped && sp.want_mat) {   // D' scratch of the geometry pre-pass: [local element][pair][64]
    const size_t need = (size_t)base.nelem * sp.l.npairs * 64;
    if ((rc = Pl->d_sf3_dprime.reserve(need))) return rc;
    sp.dprime = Pl->d_sf3_dprime.get();
  }
  const dim3 ggrid((unsigned)base.ax[0].ew, (unsigned)base.ax[1].ew, (unsigned)base.ax[2].ew);
  if (base.ax[1].ew > 65535 || base.ax[2].ew > 65535) return nope("element box too large for a 3-D grid");
  if (mapped && sp.want_mat) {          // geometry pre-pass: D' for the matrix kernel (+ the element vectors on the way)
    sf3_geom_kernel<<<ggrid, 64, 0, Pl->stream>>>(sp);
    PC_CUDA(cudaGetLastError());
    Pl->launches++;
  } else if (sp.want_vec && NV > 0 && base.ax[1].ew <= 65535 && base.ax[2].ew <= 65535) {   // vector only: the lean vector kernel (pc_quadv.cuh)
    const dim3 grid3((unsigned)base.ax[0].ew, (unsigned)base.ax[1].ew, (unsigned)base.ax[2].ew);
    if (mapped) quad_vec3_kernel<3, true><<<grid3, 64, 0, Pl->stream>>>(sp);
    else quad_vec3_kernel<3, false><<<grid3, 64, 0, Pl->stream>>>(sp);
    PC_CUDA(cudaGetLastError());
    Pl->launches++;
  } else if (sp.want_vec) {
    sf3_geom_kernel<<<ggrid, 64, 0, Pl->stream>>>(sp);
    PC_CUDA(cudaGetLastError());
    Pl->launches++;
  }
  if (sp.want_mat) {
    const int blocks = std::min(sp.npencils * sp.nseg, Pl->num_sms);
    const SF3RSmem layr(sp.l.npairs, mapped ? 1 : 0);
    if (smooth0 && Pl->sf3_variant == 0 && (size_t)layr.total * 8 <= 227 * 1024) {   // rows carried in the DMMA accumulators
      const size_t smem = (size_t)layr.total * 8;
      auto same = [&](const SF3RStruct& S) {      // exact match of the run-time lists with a compiled-in structure
        if (sp.l.ng2 != S.ng2 || sp.l.ng1 != S.ng1 || sp.l.npairs != S.npairs) return false;
        for (int k = 0; k <= S.ng2; k++) if (sp.l.g2_first[k] != S.g2_first[k]) return false;
        for (int k = 0; k < S.ng2; k++) if (sp.l.g2_oo2[k] != S.g2_oo2[k]) return false;
        for (int k = 0; k <= S.ng1; k++) if (sp.l.g1_first[k] != S.g1_first[k]) return false;
        for (int k = 0; k < S.ng1; k++) if (sp.l.g1_oo1[k] != S.g1_oo1[k]) return false;
        for (int k = 0; k < S.npairs; k++) if (sp.l.pair_oo0[k] != S.pair_oo0[k]) return false;
        return true;
      };
      if (getenv("PETIGA_SF3_DUMP")) {
        printf("sf3 lists: mapped=%d ng2=%d ng1=%d npairs=%d\n g2_first:", (int)mapped, sp.l.ng2, sp.l.ng1, sp.l.npairs);
        for (int k = 0; k <= sp.l.ng2; k++) printf(" %d", sp.l.g2_first[k]);
        printf("\n g2_oo2:"); for (int k = 0; k < sp.l.ng2; k++) printf(" %d", sp.l.g2_oo2[k]);
        printf("\n g1_first:"); for (int k = 0; k <= sp.l.ng1; k++) printf(" %d", sp.l.g1_first[k]);
        printf("\n g1_oo1:"); for (int k = 0; k < sp.l.ng1; k++) printf(" %d", sp.l.g1_oo1[k]);
        printf("\n pair_oo0:"); for (int k = 0; k < sp.l.npairs; k++) printf(" %d", sp.l.pair_oo0[k]);
        printf("\n pair_s/t:"); for (int k = 0; k < sp.l.npairs; k++) printf(" (%d,%d)", sp.l.pair_s[k], sp.l.pair_t[k]);
        printf("\n"); fflush(stdout);
      }
      const int fs = Pl->sf3_static == 0 ? 0 : (!mapped && same(k3rStructDiag)) ? 1 : (mapped && same(k3rStructFull)) ? 2 : 0;
#define SF3R_LAUNCH(FS_) { PC_CUDA(cudaFuncSetAttribute(quad_sf3r_kernel<FS_>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
                           quad_sf3r_kernel<FS_><<<blocks, k3rThreads, smem, Pl->stream>>>(sp); }
      if (fs == 1) SF3R_LAUNCH(1) else if (fs == 2) SF3R_LAUNCH(2) else SF3R_LAUNCH(0)
#undef SF3R_LAUNCH
      Pl->last_sf3_variant = 0;
      Pl->last_sf3_static = fs;
    } else {
      const SF3Smem lay(sp.l.npairs, mapped ? 1 : 0);
      const size_t smem = (size_t)lay.total * 8;
      if (smem > 227 * 1024) return nope("shared memory");
      PC_CUDA(cudaFuncSetAttribute(quad_sf3_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      quad_sf3_kernel<<<blocks, k3Threads, smem, Pl->stream>>>(sp);
      Pl->last_sf3_variant = 1;
    }
    PC_CUDA(cudaGetLastError());
    Pl->launches++;
  }
  // FP64 operations executed per element: DMMA count x 512, plus the FMA stages of the geometry group
  const double dmmas = NA > 0 ? 8.0 * sp.l.npairs + 16.0 * sp.l.ng1 + 64.0 * sp.l.ng2 : 0.0;
  const double geo = (mapped ? 2.0 * 4 * (384 + 576 + 768) + 200.0 * 64 : 0.0) + (NV > 0 ? 2.0 * 4 * sp.l.NT * (64 + 64 + 64) : 0.0) + (NA > 0 ? 2.0 * sp.l.npairs * 64 : 0.0);
  Pl->last_flops = (double)base.nelem * (dmmas * 512.0 + geo);
  return 0;
}

}  // namespace pc
