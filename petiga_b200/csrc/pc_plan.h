// pc_plan.h -- the plan object behind the C ABI (internal).
#pragma once
#include <cuda_runtime.h>

#include <string>
#include <vector>

#include "pc_device.h"

struct petiga_cuda_plan {
  pc::Layout L;
  int device = 0;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  void* nccl = nullptr;           // ncclComm_t
  int order = 1;

  // host copies needed later
  std::vector<double> detJac_h[3];
  std::vector<int> first_h[3];

  // device tables
  pc::DevAxis dax[3];
  std::vector<void*> allocs;      // everything cudaMalloc'ed by the plan (freed on destroy)
  int* d_localrow = nullptr;
  int* d_staterow = nullptr;      // collocation plans: ghost box -> state row (Layout::staterow)
  int64_t* d_rowbase = nullptr;
  int* d_rowG[3] = {nullptr, nullptr, nullptr};
  int* d_first[3] = {nullptr, nullptr, nullptr};
  int* d_own[3] = {nullptr, nullptr, nullptr};
  int* d_box_ls[3] = {nullptr, nullptr, nullptr};
  int* d_box_lw[3] = {nullptr, nullptr, nullptr};
  int* d_rank_start = nullptr;
  // 1-D element matrices for the separable path: [comp pair][nel][nen][nen]
  double* d_kron1d[3] = {nullptr, nullptr, nullptr};
  double* d_kronrow[3] = {nullptr, nullptr, nullptr};   // 1-D global banded matrices [4][nnp][kMaxW]
  double* d_sfpp[3] = {nullptr, nullptr, nullptr};      // pair-product tables of the sum-factorised kernel
  double* d_sf3pp[3] = {nullptr, nullptr, nullptr};     // the same products in the fragment layout of the third-generation kernel
  double* d_solve_work = nullptr; size_t solve_work_cap = 0;     // pc_solve.cu: r, z, p, Ap, 1/diag, reduction partials, scalars
  double* d_solve_xfull = nullptr; size_t solve_xfull_cap = 0;   // full-length operand of a distributed matrix-vector product
  double* d_gmres_work = nullptr; size_t gmres_work_cap = 0;     // pc_solve.cu GMRES: Krylov basis, w, z, 1/diag, partials, Hessenberg, rotations
  double* d_sf3_dprime = nullptr; size_t sf3_dprime_cap = 0;   // D'[element][pair][64] of the geometry pre-pass (mapped geometry)

  // pattern (owned by the plan), per block mode
  int* d_rowptr[2] = {nullptr, nullptr};
  int* d_colidx[2] = {nullptr, nullptr};

  // geometry / bc / state
  double* d_X = nullptr;
  double* d_W = nullptr;
  double* d_fixtable = nullptr;
  double* d_bnd_value[3][2] = {{nullptr, nullptr}, {nullptr, nullptr}, {nullptr, nullptr}};   // IGABasis.bnd_value on the device
  double bnd_point[3][2] = {{0, 0}, {0, 0}, {0, 0}};
  int visit[3][2] = {{0, 0}, {0, 0}, {0, 0}};            // IGASetBoundaryForm flags
  double* d_face_dS[3][2] = {{nullptr, nullptr}, {nullptr, nullptr}, {nullptr, nullptr}};   // BoundaryArea factors of mapped faces with loads
  long face_version[3][2] = {{-1, -1}, {-1, -1}, {-1, -1}};
  petiga_cuda_bc bc;
  bool has_bc = false;
  // unified local buffers (multi-rank) and exchange staging
  double* d_ghost_values = nullptr; size_t ghost_values_cap = 0;
  double* d_rhs_loc = nullptr;     // [nloc*dof]
  double* d_U_loc = nullptr;       // [nloc*dof] (collocation: [nstate*dof])
  double* d_V_loc = nullptr;
  double* d_W_loc = nullptr;
  double* d_recv = nullptr; size_t recv_cap = 0;
  int* d_recv_rows = nullptr;      // concatenated recv row lists (collocation: the state_recv lists)
  int64_t* d_recv_off = nullptr;   // same indexing: block offset of each listed row inside its peer's slab
  std::vector<size_t> recv_row_off;
  // host staging for *_host entry points
  double* h_pinned = nullptr; size_t h_pinned_cap = 0;
  double* d_values_own = nullptr; size_t values_own_cap = 0;   // device arrays used by compute_host
  double* d_rhs_own = nullptr;
  double* d_U_own = nullptr;
  double* d_V_own = nullptr;
  double* d_scalar = nullptr; size_t scalar_cap = 0;   // [0,8): result, then per-CTA partials of compute_scalar

  struct Slot { int form = -1; double prm[pc::kMaxPrm] = {0}; } slots[PETIGA_NSLOTS];
  int path = PETIGA_PATH_AUTO;
  int scatter = 0;
  std::vector<unsigned char> kron_cache;   // cached parameter block of the separable path
  int kron_cache_slot = -1, kron_cache_block = -1;
  long kron_cache_version = -1, config_version = 0;   // bumped by form_select / set_bc / set_geometry
  int kron_minb_rows = 100;       // separable path, dof 1: axis-0 rows per pencil from which the 3-CTA instantiation is used
  int kron_bulk = 0;              // separable path, dof 1: 1 = rows staged in shared memory and written by cp.async.bulk stores
  int sf3_variant = 0;            // third-generation kernel: 0 = register-carried rows where the axis-0 rows advance one per element, 1 = shared-memory window always
  int last_sf3_variant = 0;
  int sf3_static = 1, last_sf3_static = 0;   // 1: use the compiled-in form structure when the run-time lists match it (0: always interpret)
  int quad_impl = -1;             // -1 = choose by element size, 0 = sum-factorised kernel, 1 = pair-loop kernel
  // stats
  long launches = 0;
  int last_path = 0;
  int last_impl = 0;
  double last_kernel_ms = 0;
  double last_flops = 0;          // FP64 operations the last quadrature launch executes (analytic count by its launcher)
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  int num_sms = 148;
};

namespace pc {
void set_error(const std::string& msg);
void nvtx_push(int slot);   // NVTX range named after the IGACompute* driver the slot stands for (no-op without libnvToolsExt)
void nvtx_pop();
int cuda_fail(cudaError_t e, const char* what);
#define PC_CUDA(call)                                              \
  do {                                                             \
    cudaError_t _e = (call);                                       \
    if (_e != cudaSuccess) return pc::cuda_fail(_e, #call);        \
  } while (0)

// quadrature path (pc_quad.cu)
int launch_quadrature(petiga_cuda_plan* P, const KParams& base);      // v1: pair loop as one register-tiled contraction
int launch_quadrature_sf(petiga_cuda_plan* P, const KParams& base);   // v2: sum-factorised
int launch_quadrature_vec3(petiga_cuda_plan* P, const KParams& base); // vector-only sum factorisation (3-D, dof 1, p = 2..4)
int launch_quadrature_sf3(petiga_cuda_plan* P, const KParams& base);  // v3: persistent, warp-specialised, DMMA (3-D, p = 3, dof 1)
int launch_quadrature_gen(petiga_cuda_plan* P, const KParams& base);  // generic runtime-degree kernel (pc_quadg.cu); also the face mode
// separable path (pc_kron.cu)
bool kron_applicable(const petiga_cuda_plan* P, int slot, int form);
int launch_kronecker(petiga_cuda_plan* P, int slot, int block, double* values, double* rhs);
// ghost exchange (pc_comm.cu)
int exchange_ghost_rows(petiga_cuda_plan* P, int block, double* values, double* rhs, bool mat, bool vec);
// state halo: U_loc = the owned part, then the runs of `ghost` received from their owners; `owned` lists what each neighbour reads
// and must be the lists uploaded to d_recv_rows (Galerkin plans: L.send / L.recv; collocation plans: L.state_send / L.state_recv)
int halo_state(petiga_cuda_plan* P, const std::vector<Layout::Peer>& ghost, const std::vector<Layout::Recv>& owned, const double* U_own,
               double* U_loc);
int nccl_load();
int allgather_owned(petiga_cuda_plan* P, const double* owned, double* full);
int allreduce_sum(petiga_cuda_plan* P, double* d_buf, int n);
void nvtx_push(const char* name);
// IGAFormBC of every face as the element fix-up reads it: the values and, with loads, the Neumann loads of fields < dof
// (pc_api.cu).  out must be zeroed; it stays so when no boundary condition is set.  Each caller derives its own any_bc.
void fill_fix_sides(const petiga_cuda_plan* P, bool loads, FixSide out[3][2]);
// collocation rows (pc_colloc.cu): every value of the owned rows and the owned right-hand side, written once
int launch_collocation(petiga_cuda_plan* P, int slot, int form, double* values, double* rhs);
// the Bratu collocation slots (Function/Jacobian, IFunction/IJacobian); U, V in the state numbering (Layout::staterow)
int launch_collocation_state(petiga_cuda_plan* P, int slot, const double* U, const double* V, double shift, double* values, double* rhs);
// boundary-integral pass (pc_bnd.cu)
int launch_boundary_pass(petiga_cuda_plan* P, int slot, int form, const double* prm, double* rhs, bool apply_fix);
}  // namespace pc
