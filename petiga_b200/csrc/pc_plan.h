// pc_plan.h -- the plan object behind the C ABI (internal).
#pragma once
#include <cuda_runtime.h>

#include <string>
#include <vector>

#include "pc_device.h"

namespace pc {
void set_error(const std::string& msg);
int cuda_fail(cudaError_t e, const char* what);
#define PC_CUDA(call)                                              \
  do {                                                             \
    cudaError_t _e = (call);                                       \
    if (_e != cudaSuccess) return pc::cuda_fail(_e, #call);        \
  } while (0)

// Sole owner of one device allocation of n elements of T; non-empty means allocated.  It frees on the current device, so whoever
// drops one makes the owning device current first.  reserve() is grow-only: it frees before it allocates, so a regrow never holds
// two buffers at once, and the contents are undefined after it.  A failed reserve() leaves the buffer empty.
template <typename T>
class DevBuf {
 public:
  DevBuf() = default;
  DevBuf(DevBuf&& o) noexcept : p_(o.p_), n_(o.n_) { o.p_ = nullptr; o.n_ = 0; }
  DevBuf& operator=(DevBuf&& o) noexcept {
    if (this != &o) { reset(); p_ = o.p_; n_ = o.n_; o.p_ = nullptr; o.n_ = 0; }
    return *this;
  }
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  ~DevBuf() { reset(); }
  T* get() const { return p_; }
  size_t size() const { return n_; }
  explicit operator bool() const { return p_ != nullptr; }
  void reset() {
    if (p_) cudaFree(p_);
    p_ = nullptr;
    n_ = 0;
  }
  int reserve(size_t n) {
    if (p_ && n <= n_) return 0;
    reset();
    if (n == 0) n = 1;
    void* d = nullptr;
    PC_CUDA(cudaMalloc(&d, n * sizeof(T)));
    p_ = static_cast<T*>(d);
    n_ = n;
    return 0;
  }
  // reserve(n), then n elements from the host on `stream` (none when src is NULL)
  int upload(const T* src, size_t n, cudaStream_t stream) {
    int rc = reserve(n);
    if (rc) return rc;
    if (src) PC_CUDA(cudaMemcpyAsync(p_, src, n * sizeof(T), cudaMemcpyHostToDevice, stream));
    return 0;
  }

 private:
  T* p_ = nullptr;
  size_t n_ = 0;
};
}  // namespace pc

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

  // device tables; every buffer the plan allocates is owned by one DevBuf member and freed with the plan.  Tables built on first
  // use (kronrow, sfpp, sf3pp, the pattern) are complete when non-empty and never move: kron_cache keeps pointers into kronrow.
  struct AxisTables {
    pc::DevBuf<double> value, weight, point, detJac;
    pc::DevBuf<int> offset, W, lo, simple;
    pc::DevBuf<uint32_t> seg;
    pc::DevBuf<int> rowG, first, own, box_ls, box_lw;
    pc::DevBuf<double> kronrow;   // 1-D global banded matrices [4][nnp][kMaxW] of the separable path, then mv, lsum, rsum, nsup
    pc::DevBuf<double> sfpp;      // pair-product tables of the sum-factorised kernel
    pc::DevBuf<double> sf3pp;     // the same products in the fragment layout of the third-generation kernel
  } d_ax[3];
  pc::DevAxis dax[3];             // kernel view of d_ax[d]
  pc::DevBuf<int> d_localrow;
  pc::DevBuf<int> d_staterow;     // collocation plans: ghost box -> state row (Layout::staterow)
  pc::DevBuf<int64_t> d_rowbase;
  pc::DevBuf<int> d_rank_start;
  pc::DevBuf<double> d_solve_work;    // pc_solve.cu: r, z, p, Ap, 1/diag, reduction partials, scalars
  pc::DevBuf<double> d_solve_xfull;   // full-length operand of a distributed matrix-vector product
  pc::DevBuf<double> d_gmres_work;    // pc_solve.cu GMRES: Krylov basis, w, z, 1/diag, partials, Hessenberg, rotations
  pc::DevBuf<double> d_sf3_dprime;    // D'[element][pair][64] of the geometry pre-pass (mapped geometry)

  // pattern (owned by the plan), per block mode
  pc::DevBuf<int> d_rowptr[2];
  pc::DevBuf<int> d_colidx[2];

  // geometry / bc / state
  pc::DevBuf<double> d_X;
  pc::DevBuf<double> d_W;
  pc::DevBuf<double> d_fixtable;
  pc::DevBuf<double> d_bnd_value[3][2];   // IGABasis.bnd_value on the device
  double bnd_point[3][2] = {{0, 0}, {0, 0}, {0, 0}};
  int visit[3][2] = {{0, 0}, {0, 0}, {0, 0}};            // IGASetBoundaryForm flags
  pc::DevBuf<double> d_face_dS[3][2];     // BoundaryArea factors of mapped faces with loads
  long face_version[3][2] = {{-1, -1}, {-1, -1}, {-1, -1}};
  petiga_cuda_bc bc;
  bool has_bc = false;
  // unified local buffers (multi-rank) and exchange staging
  pc::DevBuf<double> d_ghost_values;
  pc::DevBuf<double> d_rhs_loc;   // [nloc*dof]
  pc::DevBuf<double> d_U_loc;     // [nloc*dof] (collocation: [nstate*dof])
  pc::DevBuf<double> d_V_loc;
  pc::DevBuf<double> d_W_loc;
  pc::DevBuf<double> d_recv;
  pc::DevBuf<int> d_recv_rows;        // concatenated recv row lists (collocation: the state_recv lists)
  pc::DevBuf<int64_t> d_recv_off;     // same indexing: block offset of each listed row inside its peer's slab
  std::vector<size_t> recv_row_off;
  pc::DevBuf<double> d_values_own;   // device arrays used by compute_host
  pc::DevBuf<double> d_rhs_own;
  pc::DevBuf<double> d_U_own;
  pc::DevBuf<double> d_V_own;
  pc::DevBuf<double> d_scalar;       // [0,8): result, then per-CTA partials of compute_scalar

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
void nvtx_push(int slot);   // NVTX range named after the IGACompute* driver the slot stands for (no-op without libnvToolsExt)
void nvtx_pop();

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
