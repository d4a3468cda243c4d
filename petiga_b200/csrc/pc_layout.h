// pc_layout.h -- host-side integer layout of one rank: numbering, CSR row bases, closed-form column
// positions and the neighbour exchange lists.  Pure C++ (no CUDA) so that it can be unit-tested on a CPU
// box; the device plan uploads these tables unchanged.
//
// Reference semantics reproduced here (bit-exact integer work):
//   * box partition            src/petigapart.c:170-202 (IGA_Distribute), src/petiga.c:1160-1209
//   * global numbering / lgmap src/petigagrid.c:98-171,185-228
//   * row stencil              src/petigamat.c:197-267 (Stencil, ColumnIndices), both branches
//   * collocation boxes        the element box is the owned node box, the ghost box the union of the owned rows' stencils;
//                              the state halo of that ghost box (staterow, state_send, state_recv)
// What is new: instead of searching a sorted row per inserted value (MatSetValues), the position of
// column B inside row A is computed in closed form from three per-axis tables (see col_position()).
#pragma once
#include <cstdint>
#include <string>
#include <vector>

#include "../../include/petiga_cuda.h"

#ifdef __CUDACC__
#define PC_HOST_DEVICE __host__ __device__ __forceinline__
#else
#define PC_HOST_DEVICE inline
#endif

namespace pc {

constexpr int kMaxP = 8;              // tuned kernels are instantiated for p = 1..4, the generic kernel (pc_quadg.cuh) runs p <= 8
constexpr int kMaxW = 2 * kMaxP + 1;  // widest 1-D stencil

struct AxisLayout {
  int p = 0, m = 1, nel = 1, nnp = 1, periodic = 0, nqp = 1;
  int P = 1, r = 0;                       // processor grid size / my coordinate along this axis
  int es = 0, ew = 1;                     // my element box
  int ls = 0, lw = 1, gs = 0, gw = 1;     // my owned / ghost node box (unwrapped coordinates)
  std::vector<int> first, last;           // [nnp]  Stencil() of every node
  std::vector<int> own;                   // [nnp]  owner processor coordinate of every node
  std::vector<int> box_es, box_ew, box_ls, box_lw, box_gs, box_gw;   // [P] boxes of every coordinate
  // indexed by ghost coordinate g in [0, gw):
  std::vector<int> wrapped;               // node index after periodic wrap
  std::vector<int> W, lo;                 // row width; lo = (unwrapped row coordinate) - first
  std::vector<int> simple;                // 1 when the row's columns are already in storage order (one owner, no wrap)
  std::vector<uint32_t> seg;              // [gw][kMaxW]: B | S<<8 | L<<16 for column offset c (see below)
};

struct Layout {
  int dim = 1, dof = 1, rank = 0, nranks = 1;
  int collocation = 0;                    // rows are the owned nodes only: no ghost rows, nothing to exchange
  AxisLayout ax[3];
  int nown = 0;                           // owned nodes
  int nghostrows = 0;                     // distinct nodes in the ghost box owned by other ranks
  int nloc = 0;                           // nown + nghostrows = rows of the unified local buffer
  int64_t nnz_own = 0, nnz_loc = 0;       // blocks in owned rows / in owned+ghost rows
  std::vector<int> rank_start;            // [nranks+1] first global node of every rank
  std::vector<int> localrow;              // [gw0*gw1*gw2] ghost-box node -> local row id (collocation: -1 for nodes of other ranks)
  std::vector<int> lgmap;                 // [gw0*gw1*gw2] ghost-box node -> global node
  std::vector<int64_t> rowbase;           // [nloc+1] block offset of every local row (owned rows first)
  std::vector<int> rowW[3];               // [nloc] per-axis widths of every local row
  std::vector<int> rowG[3];               // [nloc] per-axis *node* coordinate (wrapped) of every local row
  // ghost-row exchange: my ghost rows are grouped by owner, ascending owner-local index
  struct Peer { int rank; int first_row; int nrows; int64_t first_block; int64_t nblocks; };
  std::vector<Peer> send;                 // ghost rows I hold for `rank`  (contiguous local rows)
  struct Recv { int rank; std::vector<int> rows; int64_t nblocks; };
  std::vector<Recv> recv;                 // my owned rows that `rank` holds as ghost rows, in its order
  // collocation state halo (empty on Galerkin layouts, whose halo uses send/recv): the kernels read U at every node of the
  // ghost box, and the nodes of other ranks are numbered after the owned rows, ascending global id (one run per owner)
  std::vector<int> staterow;              // [gw0*gw1*gw2] ghost-box node -> state row (owned: its row; foreign: nown + t)
  int nstate = 0;                         // nown + foreign nodes of the ghost box
  std::vector<Peer> state_send;           // the run of foreign nodes that `rank` owns (first_row, nrows; no blocks)
  std::vector<Recv> state_recv;           // my owned rows inside `rank`'s ghost box, in its order (nblocks 0)
  std::string error;
};

// Builds the layout; returns 0 or a PETIGA_CUDA_ERR_* code with L.error set.
int build_layout(const petiga_cuda_space& sp, int rank, int nranks, Layout& L);

// closed-form position (in blocks, relative to the row base) of a column inside its row from the seg entries s0, s1, s2 of
// the column's per-axis offsets and the row widths W0, W1 of axes 0 and 1.  Shared by the host and the quadrature kernels.
PC_HOST_DEVICE int seg_position(uint32_t s0, uint32_t s1, uint32_t s2, int W0, int W1) {
  const int Bi = s0 & 255, Si = (s0 >> 8) & 255, Li = (s0 >> 16) & 255;
  const int Bj = s1 & 255, Sj = (s1 >> 8) & 255, Lj = (s1 >> 16) & 255;
  const int Bk = s2 & 255, Sk = (s2 >> 8) & 255, Lk = (s2 >> 16) & 255;
  return Bk * W1 * W0 + Sk * (Bj * W0 + Sj * Bi) + (Lk * Sj + Lj) * Si + Li;
}

// seg_position of the column with per-axis offsets c[d] (c = unwrapped column coordinate - first(row)) inside the row with
// per-axis ghost coordinates g[d].
inline int64_t col_position(const Layout& L, const int g[3], const int c[3]) {
  return seg_position(L.ax[0].seg[g[0] * kMaxW + c[0]], L.ax[1].seg[g[1] * kMaxW + c[1]], L.ax[2].seg[g[2] * kMaxW + c[2]],
                      L.ax[0].W[g[0]], L.ax[1].W[g[1]]);
}

// Host generation of the owned-row pattern (tests, small meshes).  block=0 expands to scalar AIJ rows.
int host_pattern(const Layout& L, int block, std::vector<int>& rowptr, std::vector<int>& colidx);

}  // namespace pc
