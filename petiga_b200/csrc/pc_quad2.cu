// pc_quad2.cu -- component lists and launcher of the sum-factorised quadrature kernel (pc_quad2.cuh).
#include <algorithm>
#include <cstring>
#include <vector>

#include "pc_plan.h"
#include "pc_quad2.cuh"

namespace pc {

// ------------------------------------------------------------------------------------------------------------
// sum-factorised kernel (pc_quad2.cuh): component lists and launch
template <int DIM, int DOF>
void host_matrix_pattern(int form, int slot, const double* prm, const FormInfo& fi, std::vector<char>& pat, int& ijmask, std::vector<double>& Cout) {
  const int NA = fi.mc1 - fi.mc0;
  pat.assign((size_t)std::max(NA * NA, 1), 0);
  ijmask = 0;
  if (NA == 0) return;
  if (fi.per_qp) {   // coefficients depend on the point: assume every entry can be nonzero
    std::fill(pat.begin(), pat.end(), 1);
    ijmask = (1 << (DOF * DOF)) - 1;
    return;
  }
  std::vector<double>& C = Cout;
  C.assign((size_t)DOF * DOF * NA * NA, 0.0);
  QPoint q;
  memset(&q, 0, sizeof(q));
  form_coefficients<DIM, DOF>(form, slot, prm, 0.0, 0.0, q, NA, 0, C.data(), nullptr);
  for (int ij = 0; ij < DOF * DOF; ij++)
    for (int k = 0; k < NA * NA; k++)
      if (C[(size_t)ij * NA * NA + k] != 0.0) { pat[k] = 1; ijmask |= 1 << ij; }
}

int build_sf_lists(const KParams& kp, const FormInfo& fi, bool mapped, bool rational, bool state, bool transient,
                   const std::vector<char>& cpat, int ijmask, SFLists& l) {
  memset(&l, 0, sizeof(l));
  const int dim = kp.dim, dof = kp.dof;
  const bool hasG = (kp.c1 > 1 && kp.c0 <= dim) || mapped || rational;
  const bool hasL = kp.c1 > dim + 1;
  const bool hasN = (kp.c0 == 0) || rational || (mapped && kp.needs_x);
  l.tN = -1;
  for (int d = 0; d < 3; d++) l.tG[d] = l.tL[d] = -1;
  int nt = 0;
  if (hasN) { l.tN = nt; nt++; }
  if (hasG) for (int d = 0; d < dim; d++) { l.tG[d] = nt; l.torder[nt][d] = 1; nt++; }
  if (hasL) for (int d = 0; d < dim; d++) { l.tL[d] = nt; l.torder[nt][d] = 2; nt++; }
  l.NT = nt;
  // which tensor components a physical component reaches
  auto reach = [&](int c, std::vector<int>& out) {
    out.clear();
    if (c == 0) out.push_back(l.tN);
    else if (c <= dim) {
      if (mapped) { for (int d = 0; d < dim; d++) out.push_back(l.tG[d]); } else out.push_back(l.tG[c - 1]);
      if (rational) out.push_back(l.tN);
    } else for (int d = 0; d < dim; d++) out.push_back(l.tL[d]);
  };
  // contraction pairs
  const int NA = kp.mc1 - kp.mc0;
  std::vector<char> pm((size_t)nt * nt, 0);
  std::vector<int> rs, rt;
  for (int al = 0; al < NA; al++)
    for (int be = 0; be < NA; be++) {
      if (!cpat[(size_t)al * NA + be]) continue;
      reach(al + kp.mc0, rs); reach(be + kp.mc0, rt);
      for (int s : rs) for (int t : rt) pm[(size_t)s * nt + t] = 1;
    }
  int g1key[kMaxPairs], g2key[9];
  l.npairs = l.ng1 = l.ng2 = 0;
  for (int s = 0; s < nt; s++)
    for (int t = 0; t < nt; t++) {
      if (!pm[(size_t)s * nt + t]) continue;
      if (l.npairs >= kMaxPairs) return PETIGA_CUDA_ERR_SUP;
      const int oo1 = l.torder[s][1] * 3 + l.torder[t][1], oo2 = l.torder[s][2] * 3 + l.torder[t][2];
      int g2 = -1;
      for (int k = 0; k < l.ng2; k++) if (g2key[k] == oo2) g2 = k;
      if (g2 < 0) { g2 = l.ng2; g2key[l.ng2] = oo2; l.g2_oo2[l.ng2] = (unsigned char)oo2; l.ng2++; }
      const int key = oo1 * 9 + oo2;
      int g1 = -1;
      for (int k = 0; k < l.ng1; k++) if (g1key[k] == key) g1 = k;
      if (g1 < 0) { g1 = l.ng1; g1key[l.ng1] = key; l.g1_oo1[l.ng1] = (unsigned char)oo1; l.g1_g2[l.ng1] = (unsigned char)g2; l.ng1++; }
      l.pair_s[l.npairs] = (unsigned char)s; l.pair_t[l.npairs] = (unsigned char)t; l.pair_g1[l.npairs] = (unsigned char)g1;
      l.npairs++;
    }
  {  // order the g1 groups by their g2 group so that stage B walks a contiguous range per g2
    int perm[kMaxPairs], inv[kMaxPairs], n = 0;
    for (int g2 = 0; g2 < l.ng2; g2++) {
      l.g2_first[g2] = (unsigned char)n;
      for (int g1 = 0; g1 < l.ng1; g1++) if (l.g1_g2[g1] == g2) perm[n++] = g1;
    }
    l.g2_first[l.ng2] = (unsigned char)n;
    unsigned char oo1[kMaxPairs], gg2[kMaxPairs];
    for (int k = 0; k < n; k++) { oo1[k] = l.g1_oo1[perm[k]]; gg2[k] = l.g1_g2[perm[k]]; inv[perm[k]] = k; }
    for (int k = 0; k < n; k++) { l.g1_oo1[k] = oo1[k]; l.g1_g2[k] = gg2[k]; }
    for (int k = 0; k < l.npairs; k++) l.pair_g1[k] = (unsigned char)inv[l.pair_g1[k]];
  }
  {  // order the pairs by g1 group (stage A walks a contiguous range per output) and cache their axis-0 order pair
    int perm[kMaxPairs], n = 0;
    for (int g1 = 0; g1 < l.ng1; g1++) {
      l.g1_first[g1] = (unsigned char)n;
      for (int k = 0; k < l.npairs; k++) if (l.pair_g1[k] == g1) perm[n++] = k;
    }
    l.g1_first[l.ng1] = (unsigned char)n;
    unsigned char ps[kMaxPairs], pt[kMaxPairs], pg[kMaxPairs];
    for (int k = 0; k < n; k++) { ps[k] = l.pair_s[perm[k]]; pt[k] = l.pair_t[perm[k]]; pg[k] = l.pair_g1[perm[k]]; }
    for (int k = 0; k < n; k++) {
      l.pair_s[k] = ps[k]; l.pair_t[k] = pt[k]; l.pair_g1[k] = pg[k];
      l.pair_oo0[k] = (unsigned char)(l.torder[ps[k]][0] * 3 + l.torder[pt[k]][0]);
    }
  }
  l.ijmask = ijmask;
  // fields and evaluation combos
  for (int f = 0; f < 16; f++) for (int t = 0; t < kMaxT; t++) l.ev_index[f][t] = -1;
  l.f_x0 = l.f_w = l.f_u0 = l.f_v0 = -1;
  int nf = 0;
  auto add = [&](int field, int t) -> int {
    if (t < 0 || l.ev_index[field][t] >= 0) return 0;
    if (l.nev >= kMaxEval) return 1;
    l.ev_field[l.nev] = (unsigned char)field; l.ev_t[l.nev] = (unsigned char)t; l.ev_index[field][t] = l.nev; l.nev++;
    return 0;
  };
  int bad = 0;
  if (mapped) {
    l.f_x0 = nf; nf += dim;
    for (int i = 0; i < dim; i++) {
      for (int d = 0; d < dim; d++) bad |= add(l.f_x0 + i, l.tG[d]);
      if (rational || kp.needs_x) bad |= add(l.f_x0 + i, l.tN);
    }
  }
  if (rational) {
    l.f_w = nf; nf += 1;
    bad |= add(l.f_w, l.tN);
    for (int d = 0; d < dim; d++) bad |= add(l.f_w, l.tG[d]);
  }
  if (state) {
    l.f_u0 = nf; nf += dof;
    for (int c = 0; c < dof; c++) for (int t = 0; t < nt; t++) bad |= add(l.f_u0 + c, t);
    if (transient) { l.f_v0 = nf; nf += dof; for (int c = 0; c < dof; c++) bad |= add(l.f_v0 + c, l.tN); }
  }
  l.nfields = nf;
  if (bad || nf > 16) return PETIGA_CUDA_ERR_SUP;
  return 0;
}

template void host_matrix_pattern<3, 1>(int, int, const double*, const FormInfo&, std::vector<char>&, int&, std::vector<double>&);

namespace {

template <int DIM, int P, int DOF, int NQ>
int launch_sf_nq(petiga_cuda_plan* Pl, SFParams& sp) {
  using Cfg = SFCfg<DIM, P, DOF>;
  const KParams& base = sp.k;
  const int NA = base.mc1 - base.mc0, NV = base.vc1 - base.vc0;
  const int nq[3] = {base.ax[0].nqp, base.ax[1].nqp, base.ax[2].nqp};
  const SFSmem lay(Cfg::n0, Cfg::n1, Cfg::n2, nq[0], nq[1], nq[2], DIM, DOF, sp.l, NA, NV, base.per_qp, base.c1 - base.c0);
  const size_t per = (size_t)lay.total * 8, budget = 110 * 1024, hard = 225 * 1024;
  if (per > hard) { set_error("sum-factorised kernel: element does not fit shared memory"); return PETIGA_CUDA_ERR_SUP; }
  int epb = std::max(1, 256 / Cfg::G);
  while (epb > 1 && per * epb > budget) epb--;
  sp.k.epb = epb;
  const size_t smem = per * epb;
  const int threads = ((Cfg::G * epb + 31) / 32) * 32;
  // the 64-register build only where it can run 4 CTAs per SM: one full-CTA element, default rule, four slots fit
  constexpr bool kHas4 = (Cfg::THREADS == 256 && Cfg::G == 256 && DOF == 1 && NQ > 0);
  const bool use4 = kHas4 && epb == 1 && (smem + 1024) * 4 <= 227 * 1024;
  const int blocks = (base.nelem + epb - 1) / epb;
  {  // FP64 operations this launch executes (2 per FMA), from the same lists the kernel walks
    const SFLists& l = sp.l;
    const double n0 = Cfg::n0, n1 = Cfg::n1, n2 = Cfg::n2, q0 = nq[0], q1 = nq[1], q2 = nq[2], nqp = q0 * q1 * q2, G = n0 * n0 * n1 * n1;
    int nij = 0;
    for (int ij = 0; ij < DOF * DOF; ij++) nij += (l.ijmask >> ij) & 1;
    double f = 0.0;
    if (NA > 0) f += nij * (2.0 * nqp * n0 * n0 * l.npairs + 2.0 * G * q2 * l.ng1 * q1 + G * q2 * l.ng2 * (n2 + 2.0 * n2 * n2) +
                            (sp.const_dp ? 1.0 : 2.0 * NA * NA) * l.npairs * nqp);
    f += 2.0 * l.nev * (q0 * n1 * n2 * n0 + q0 * q1 * n2 * n1 + nqp * n2);                                   // field evaluation
    if (NV > 0) f += 2.0 * DOF * l.NT * (q2 * q1 * n0 * q0 + q2 * n1 * n0 * q1 + n0 * n1 * n2 * q2) + 2.0 * nqp * DOF * l.NT * NV;
    Pl->last_flops = f * base.nelem;
  }
  auto go = [&](auto kern) -> int {
    PC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    if (blocks > 0) {
      kern<<<blocks, threads, smem, Pl->stream>>>(sp);
      PC_CUDA(cudaGetLastError());
      Pl->launches++;
    }
    return 0;
  };
  if constexpr (kHas4) { if (use4) return go(quad_sf_kernel<DIM, P, DOF, NQ, 4>); }
  return go(quad_sf_kernel<DIM, P, DOF, NQ, 1>);
}

template <int DIM, int P, int DOF>
int launch_sf(petiga_cuda_plan* Pl, const KParams& base, const FormInfo& fi) {
  SFParams sp;
  memset(&sp, 0, sizeof(sp));
  sp.k = base;
  const bool mapped = base.X != nullptr, rational = base.Wt != nullptr;
  const bool state = base.needs_state && base.U != nullptr;
  const bool transient = (base.slot == PETIGA_SLOT_IFUNCTION || base.slot == PETIGA_SLOT_IJACOBIAN);
  std::vector<char> cpat;
  std::vector<double> Cc;
  int ijmask = 0;
  host_matrix_pattern<DIM, DOF>(base.form, base.slot, base.prm, fi, cpat, ijmask, Cc);
  int rc = build_sf_lists(base, fi, mapped, rational, state, transient, cpat, ijmask, sp.l);
  if (rc) { set_error("sum-factorised kernel: too many components for this form"); return rc; }
  // per-axis pair-product tables, built once per plan (into a local buffer, kept once the build has been launched)
  for (int d = 0; d < 3; d++) {
    if (!Pl->d_ax[d].sfpp) {
      const size_t n = (size_t)base.ax[d].nel * 9 * base.ax[d].nqp * base.ax[d].nen * base.ax[d].nen;
      DevBuf<double> pp;
      if ((rc = pp.reserve(n))) return rc;
      sf_pp_kernel<<<(int)std::min<size_t>((n + 255) / 256, 4096), 256, 0, Pl->stream>>>(base.ax[d], pp.get());
      PC_CUDA(cudaGetLastError());
      Pl->launches++;
      Pl->d_ax[d].sfpp = std::move(pp);
    }
    sp.pp[d] = Pl->d_ax[d].sfpp.get();
  }
  // identity geometry + constant coefficients: D'[ij][pair] is a constant times JW
  const int NA = base.mc1 - base.mc0;
  sp.const_dp = 0;
  if (!mapped && !rational && !fi.per_qp && NA > 0 && DOF * DOF <= 9) {
    sp.const_dp = 1;
    auto phys_of = [&](int t) -> int {   // tensor component -> physical component (identity map)
      if (t == sp.l.tN) return 0;
      for (int d = 0; d < DIM; d++) if (t == sp.l.tG[d]) return 1 + d;
      return DIM + 1;
    };
    for (int ij = 0; ij < DOF * DOF; ij++)
      for (int pr = 0; pr < sp.l.npairs; pr++) {
        const int al = phys_of(sp.l.pair_s[pr]) - base.mc0, be = phys_of(sp.l.pair_t[pr]) - base.mc0;
        double c = 0.0;
        if (al >= 0 && al < NA && be >= 0 && be < NA) c = Cc[((size_t)ij * NA + al) * NA + be];
        sp.cconst[ij * kMaxPairs + pr] = c;
      }
  }
  const int nq0 = base.ax[0].nqp;
  bool def = (nq0 == P + 1);
  for (int d = 1; d < DIM; d++) def = def && base.ax[d].nqp == P + 1;
  if (def) return launch_sf_nq<DIM, P, DOF, P + 1>(Pl, sp);
  return launch_sf_nq<DIM, P, DOF, 0>(Pl, sp);
}

}  // namespace

#define SF_CASE(DIM_, P_, DOF_) \
  if (dim == DIM_ && p == P_ && dof == DOF_) return launch_sf<DIM_, P_, DOF_>(Pl, base, fi);

int launch_quadrature_sf(petiga_cuda_plan* Pl, const KParams& base) {
  const int dim = base.dim, dof = base.dof, p = base.ax[0].p;
  for (int d = 1; d < dim; d++)
    if (base.ax[d].p != p) { set_error("quadrature kernel: mixed degrees per axis are not instantiated"); return PETIGA_CUDA_ERR_SUP; }
  FormInfo fi = form_info(base.form, base.slot, dim, dof);
  SF_CASE(1, 1, 1) SF_CASE(1, 2, 1) SF_CASE(1, 3, 1) SF_CASE(1, 4, 1)
  SF_CASE(1, 1, 2) SF_CASE(1, 2, 2) SF_CASE(1, 3, 2) SF_CASE(1, 4, 2)
  SF_CASE(1, 1, 3) SF_CASE(1, 2, 3) SF_CASE(1, 3, 3) SF_CASE(1, 4, 3)
  SF_CASE(2, 1, 1) SF_CASE(2, 2, 1) SF_CASE(2, 3, 1) SF_CASE(2, 4, 1)
  SF_CASE(2, 1, 2) SF_CASE(2, 2, 2) SF_CASE(2, 3, 2) SF_CASE(2, 4, 2)
  SF_CASE(2, 1, 3) SF_CASE(2, 2, 3) SF_CASE(2, 3, 3) SF_CASE(2, 4, 3)
  SF_CASE(3, 1, 1) SF_CASE(3, 2, 1) SF_CASE(3, 3, 1) SF_CASE(3, 4, 1)
  SF_CASE(3, 1, 2) SF_CASE(3, 2, 2) SF_CASE(3, 3, 2) SF_CASE(3, 4, 2)
  SF_CASE(3, 1, 3) SF_CASE(3, 2, 3) SF_CASE(3, 3, 3) SF_CASE(3, 4, 3)
  set_error("quadrature kernel: (dim, degree, dof) combination not instantiated");
  return PETIGA_CUDA_ERR_SUP;
}


}  // namespace pc
