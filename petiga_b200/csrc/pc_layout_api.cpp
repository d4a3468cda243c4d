// pc_layout_api.cpp -- C wrappers of the host-only layout logic (see include/petiga_cuda.h, last section).
#include <cstring>
#include <new>

#include "pc_layout.h"

struct petiga_layout { pc::Layout L; };

namespace pc { void set_error(const std::string& msg); }

extern "C" {

int petiga_layout_create(petiga_layout** layout, const petiga_cuda_space* space, int rank, int nranks) {
  if (!layout || !space) return PETIGA_CUDA_ERR_ARG;
  *layout = nullptr;
  petiga_layout* l = new (std::nothrow) petiga_layout();
  if (!l) return PETIGA_CUDA_ERR_MEM;
  int rc = pc::build_layout(*space, rank, nranks, l->L);
  if (rc) { pc::set_error(l->L.error); delete l; return rc; }
  *layout = l;
  return 0;
}
int petiga_layout_destroy(petiga_layout* layout) { delete layout; return 0; }
int petiga_layout_sizes(const petiga_layout* l, int* nown, int* nghostbox, int* nloc, int64_t* nnz_own, int64_t* nnz_loc) {
  if (!l) return PETIGA_CUDA_ERR_ARG;
  if (nown) *nown = l->L.nown;
  if (nghostbox) *nghostbox = (int)l->L.lgmap.size();
  if (nloc) *nloc = l->L.nloc;
  if (nnz_own) *nnz_own = l->L.nnz_own;
  if (nnz_loc) *nnz_loc = l->L.nnz_loc;
  return 0;
}
int petiga_layout_lgmap(const petiga_layout* l, int* out) { if (!l || !out) return PETIGA_CUDA_ERR_ARG; memcpy(out, l->L.lgmap.data(), l->L.lgmap.size() * sizeof(int)); return 0; }
int petiga_layout_localrow(const petiga_layout* l, int* out) { if (!l || !out) return PETIGA_CUDA_ERR_ARG; memcpy(out, l->L.localrow.data(), l->L.localrow.size() * sizeof(int)); return 0; }
int petiga_layout_rowbase(const petiga_layout* l, int64_t* out) { if (!l || !out) return PETIGA_CUDA_ERR_ARG; memcpy(out, l->L.rowbase.data(), l->L.rowbase.size() * sizeof(int64_t)); return 0; }
int petiga_layout_pattern(const petiga_layout* l, int block, int* rowptr, int* colidx) {
  if (!l) return PETIGA_CUDA_ERR_ARG;
  std::vector<int> rp, ci;
  int rc = pc::host_pattern(l->L, block, rp, ci);
  if (rc) return rc;
  if (rowptr) memcpy(rowptr, rp.data(), rp.size() * sizeof(int));
  if (colidx) memcpy(colidx, ci.data(), ci.size() * sizeof(int));
  return 0;
}
int petiga_layout_position(const petiga_layout* l, const int ga[3], const int hb[3], int64_t* pos) {
  if (!l || !pos) return PETIGA_CUDA_ERR_ARG;
  int c[3];
  for (int d = 0; d < 3; d++) {
    const pc::AxisLayout& a = l->L.ax[d];
    if (ga[d] < 0 || ga[d] >= a.gw) return PETIGA_CUDA_ERR_ARG;
    c[d] = hb[d] - ga[d] + a.lo[ga[d]];
    if (c[d] < 0 || c[d] >= a.W[ga[d]]) return PETIGA_CUDA_ERR_ARG;
  }
  *pos = pc::col_position(l->L, ga, c);
  return 0;
}
int petiga_layout_exchange(const petiga_layout* l, int kind, int* count, int64_t* out, int capacity) {
  if (!l || !count) return PETIGA_CUDA_ERR_ARG;
  const pc::Layout& L = l->L;
  if (kind < 0 || kind > 3) return PETIGA_CUDA_ERR_ARG;
  if (kind == 0 || kind == 2) {
    const auto& S = kind == 0 ? L.send : L.state_send;
    *count = (int)S.size();
    if (out) for (int i = 0; i < *count && i < capacity; i++) { out[4*i] = S[i].rank; out[4*i+1] = S[i].first_row; out[4*i+2] = S[i].nrows; out[4*i+3] = S[i].nblocks; }
  } else {
    const auto& R = kind == 1 ? L.recv : L.state_recv;
    *count = (int)R.size();
    if (out) for (int i = 0; i < *count && i < capacity; i++) { out[4*i] = R[i].rank; out[4*i+1] = R[i].rows.empty() ? -1 : R[i].rows[0]; out[4*i+2] = (int64_t)R[i].rows.size(); out[4*i+3] = R[i].nblocks; }
  }
  return 0;
}
int petiga_layout_recv_rows(const petiga_layout* l, int peer_index, int* rows, int capacity) {
  if (!l) return PETIGA_CUDA_ERR_ARG;
  const auto& R = l->L.collocation ? l->L.state_recv : l->L.recv;   // the other list is empty
  if (peer_index < 0 || peer_index >= (int)R.size() || !rows) return PETIGA_CUDA_ERR_ARG;
  const auto& r = R[peer_index].rows;
  for (int i = 0; i < (int)r.size() && i < capacity; i++) rows[i] = r[i];
  return 0;
}
int petiga_layout_staterow(const petiga_layout* l, int* nstate, int* out) {
  if (!l) return PETIGA_CUDA_ERR_ARG;
  if (!l->L.collocation) { pc::set_error("layout_staterow: only collocation layouts have a state numbering (Galerkin: localrow)"); return PETIGA_CUDA_ERR_ARG; }
  if (nstate) *nstate = l->L.nstate;
  if (out) memcpy(out, l->L.staterow.data(), l->L.staterow.size() * sizeof(int));
  return 0;
}

}  // extern "C"
