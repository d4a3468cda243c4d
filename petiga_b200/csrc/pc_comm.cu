// pc_comm.cu -- the two exchange steps of the assembly path over NCCL (one rank per GPU):
//   (i)  ghost-row sum:  what PETSc's stash does inside MatAssemblyBegin/End and VecAssemblyBegin/End
//        (src/petigaksp.c:197-200): every rank ships the rows it integrated but does not own to their
//        owner, who adds them.  Here the ghost rows are laid out exactly like the owner's CSR rows, so a
//        message is one contiguous slab per owner and the receive side is a streaming add.
//   (ii) state halo:     VecScatter g2l of IGAGetLocalVecArray (src/petigavec.c:147-169,256-269), on the Galerkin ghost rows or
//        on the collocation ghost box (the list pair the caller passes).
// NCCL is loaded with dlopen so that the library also loads on hosts without it (single-rank use).
#include <dlfcn.h>
#include <nccl.h>

#include "pc_plan.h"

namespace pc {

namespace {
struct NcclApi {
  void* handle = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  ncclResult_t (*Send)(const void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*Recv)(void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*Broadcast)(const void*, void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*GroupStart)() = nullptr;
  ncclResult_t (*GroupEnd)() = nullptr;
  const char* (*GetErrorString)(ncclResult_t) = nullptr;
} g_nccl;

int nccl_fail(ncclResult_t r, const char* what) {
  set_error(std::string(what) + ": " + (g_nccl.GetErrorString ? g_nccl.GetErrorString(r) : "nccl error"));
  return PETIGA_CUDA_ERR_NCCL;
}
#define PC_NCCL(call)                                      \
  do {                                                     \
    ncclResult_t _r = (call);                              \
    if (_r != ncclSuccess) return nccl_fail(_r, #call);    \
  } while (0)

// values[rowbase[row]*bs2 + e] += recv[off[t] + e] for the t-th listed row; one warp per row
// off[t]: block offset of the t-th listed row inside its peer's slab (prefix sum built once at plan creation)
__global__ void add_rows_kernel(const int* __restrict__ rows, const int64_t* __restrict__ off, int nrows, const int64_t* __restrict__ rowbase,
                                int bs2, double* __restrict__ values, const double* __restrict__ recv) {
  const int wpb = blockDim.x / 32, lane = threadIdx.x & 31;
  for (int t = blockIdx.x * wpb + threadIdx.x / 32; t < nrows; t += gridDim.x * wpb) {
    const int row = rows[t];
    const int64_t b0 = rowbase[row] * bs2, n = (rowbase[row + 1] - rowbase[row]) * bs2, o = off[t] * bs2;
    for (int64_t e = lane; e < n; e += 32) values[b0 + e] += recv[o + e];
  }
}
__global__ void add_vec_rows_kernel(const int* __restrict__ rows, int nrows, int dof, int64_t off, double* __restrict__ vec,
                                    const double* __restrict__ recv) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < nrows * dof) vec[(size_t)rows[i / dof] * dof + i % dof] += recv[off + i];
}
__global__ void gather_vec_rows_kernel(const int* __restrict__ rows, int nrows, int dof, const double* __restrict__ vec, double* __restrict__ out) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < nrows * dof) out[i] = vec[(size_t)rows[i / dof] * dof + i % dof];
}
}  // namespace

int nccl_load() {
  if (g_nccl.handle) return 0;
  const char* names[] = {"libnccl.so.2", "libnccl.so"};
  void* h = nullptr;
  for (const char* n : names) { h = dlopen(n, RTLD_NOW | RTLD_GLOBAL); if (h) break; }
  if (!h) { set_error("cannot dlopen libnccl.so.2"); return PETIGA_CUDA_ERR_NCCL; }
#define LOADSYM(field, sym) *(void**)(&g_nccl.field) = dlsym(h, sym); if (!g_nccl.field) { set_error("missing NCCL symbol " sym); return PETIGA_CUDA_ERR_NCCL; }
  LOADSYM(GetUniqueId, "ncclGetUniqueId") LOADSYM(CommInitRank, "ncclCommInitRank") LOADSYM(CommDestroy, "ncclCommDestroy")
  LOADSYM(Send, "ncclSend") LOADSYM(Recv, "ncclRecv") LOADSYM(GroupStart, "ncclGroupStart") LOADSYM(GroupEnd, "ncclGroupEnd")
  LOADSYM(GetErrorString, "ncclGetErrorString") LOADSYM(AllReduce, "ncclAllReduce") LOADSYM(Broadcast, "ncclBroadcast")
#undef LOADSYM
  g_nccl.handle = h;
  return 0;
}

// MPI_Allreduce(SUM) of IGAComputeScalar (src/petigacomp.c:90), in place on the plan's stream
int allreduce_sum(petiga_cuda_plan* P, double* d_buf, int n) {
  if (!P->nccl) { set_error("multi-rank plan without an NCCL communicator"); return PETIGA_CUDA_ERR_ORDER; }
  int rc = nccl_load();
  if (rc) return rc;
  PC_NCCL(g_nccl.AllReduce(d_buf, d_buf, (size_t)n, ncclDouble, ncclSum, (ncclComm_t)P->nccl, P->stream));
  P->launches += 1;
  return 0;
}

// every rank's owned slice into a full-length vector in the global (rank-major) numbering: the operand gather of a distributed
// matrix-vector product (VecScatter of MatMult_MPIAIJ); one grouped broadcast per owner, since the slices differ in length
int allgather_owned(petiga_cuda_plan* P, const double* owned, double* full) {
  const Layout& L = P->L;
  if (!P->nccl) { set_error("multi-rank plan without an NCCL communicator"); return PETIGA_CUDA_ERR_ORDER; }
  int rc = nccl_load();
  if (rc) return rc;
  ncclComm_t comm = (ncclComm_t)P->nccl;
  ncclResult_t gr = g_nccl.GroupStart();
  if (gr != ncclSuccess) return nccl_fail(gr, "ncclGroupStart");
  for (int r = 0; r < L.nranks && gr == ncclSuccess; r++) {
    const size_t off = (size_t)L.rank_start[r] * L.dof, cnt = (size_t)(L.rank_start[r + 1] - L.rank_start[r]) * L.dof;
    gr = g_nccl.Broadcast(r == L.rank ? owned : full + off, full + off, cnt, ncclDouble, r, comm, P->stream);
  }
  ncclResult_t ge = g_nccl.GroupEnd();
  if (gr != ncclSuccess) return nccl_fail(gr, "ncclBroadcast (operand gather)");
  if (ge != ncclSuccess) return nccl_fail(ge, "ncclGroupEnd");
  P->launches++;
  return 0;
}

int exchange_ghost_rows(petiga_cuda_plan* P, int block, double* values, double* rhs, bool mat, bool vec) {
  (void)block;
  const Layout& L = P->L;
  if (!P->nccl) { set_error("multi-rank plan without an NCCL communicator"); return PETIGA_CUDA_ERR_ORDER; }
  int rc = nccl_load();
  if (rc) return rc;
  ncclComm_t comm = (ncclComm_t)P->nccl;
  const int bs2 = L.dof * L.dof, dof = L.dof;
  // staging: [matrix slabs per recv peer][vector slabs per recv peer]
  size_t total = 0;
  std::vector<size_t> moff(L.recv.size()), voff(L.recv.size());
  for (size_t i = 0; i < L.recv.size(); i++) { moff[i] = total; if (mat) total += (size_t)L.recv[i].nblocks * bs2; }
  for (size_t i = 0; i < L.recv.size(); i++) { voff[i] = total; if (vec) total += L.recv[i].rows.size() * dof; }
  if ((rc = P->d_recv.reserve(total))) return rc;
  // a failed Send/Recv must not leave the NCCL group open (ADVICE r1): close it, then report
  ncclResult_t gr = g_nccl.GroupStart();
  if (gr != ncclSuccess) return nccl_fail(gr, "ncclGroupStart");
  auto post = [&](ncclResult_t r) { if (gr == ncclSuccess && r != ncclSuccess) gr = r; };
  for (const auto& s : L.send) {
    if (mat) post(g_nccl.Send(P->d_ghost_values.get() + (size_t)(s.first_block - L.nnz_own) * bs2, (size_t)s.nblocks * bs2, ncclDouble, s.rank, comm, P->stream));
    if (vec) post(g_nccl.Send(P->d_rhs_loc.get() + (size_t)s.first_row * dof, (size_t)s.nrows * dof, ncclDouble, s.rank, comm, P->stream));
  }
  for (size_t i = 0; i < L.recv.size(); i++) {
    const auto& r = L.recv[i];
    if (mat) post(g_nccl.Recv(P->d_recv.get() + moff[i], (size_t)r.nblocks * bs2, ncclDouble, r.rank, comm, P->stream));
    if (vec) post(g_nccl.Recv(P->d_recv.get() + voff[i], r.rows.size() * dof, ncclDouble, r.rank, comm, P->stream));
  }
  ncclResult_t ge = g_nccl.GroupEnd();
  if (gr != ncclSuccess) return nccl_fail(gr, "ncclSend/ncclRecv (ghost rows)");
  if (ge != ncclSuccess) return nccl_fail(ge, "ncclGroupEnd");
  P->launches += 1;
  for (size_t i = 0; i < L.recv.size(); i++) {
    const auto& r = L.recv[i];
    const int n = (int)r.rows.size();
    const int* rows = P->d_recv_rows.get() + P->recv_row_off[i];
    if (mat) {   // per-row offsets inside the slab were uploaded once by petiga_cuda_plan_create: no host work, no sync here
      add_rows_kernel<<<std::max(1, std::min((n + 7) / 8, P->num_sms * 8)), 256, 0, P->stream>>>(rows, P->d_recv_off.get() + P->recv_row_off[i], n, P->d_rowbase.get(), bs2,
                                                                                               values, P->d_recv.get() + moff[i]);
      PC_CUDA(cudaGetLastError());
      P->launches++;
    }
    if (vec) {
      add_vec_rows_kernel<<<(n * dof + 255) / 256, 256, 0, P->stream>>>(rows, n, dof, (int64_t)voff[i], P->d_rhs_loc.get(), P->d_recv.get());
      PC_CUDA(cudaGetLastError());
      P->launches++;
    }
  }
  if (vec) PC_CUDA(cudaMemcpyAsync(rhs, P->d_rhs_loc.get(), (size_t)L.nown * dof * sizeof(double), cudaMemcpyDeviceToDevice, P->stream));
  return 0;
}

int halo_state(petiga_cuda_plan* P, const std::vector<Layout::Peer>& ghost, const std::vector<Layout::Recv>& owned, const double* U_own,
               double* U_loc) {
  const Layout& L = P->L;
  if (!P->nccl) { set_error("multi-rank plan without an NCCL communicator"); return PETIGA_CUDA_ERR_ORDER; }
  int rc = nccl_load();
  if (rc) return rc;
  ncclComm_t comm = (ncclComm_t)P->nccl;
  const int dof = L.dof;
  PC_CUDA(cudaMemcpyAsync(U_loc, U_own, (size_t)L.nown * dof * sizeof(double), cudaMemcpyDeviceToDevice, P->stream));
  size_t total = 0;
  std::vector<size_t> off(owned.size());
  for (size_t i = 0; i < owned.size(); i++) { off[i] = total; total += owned[i].rows.size() * dof; }
  if ((rc = P->d_recv.reserve(total))) return rc;
  for (size_t i = 0; i < owned.size(); i++) {   // owners pack the rows their neighbours see as ghosts
    const int n = (int)owned[i].rows.size();
    gather_vec_rows_kernel<<<(n * dof + 255) / 256, 256, 0, P->stream>>>(P->d_recv_rows.get() + P->recv_row_off[i], n, dof, U_own, P->d_recv.get() + off[i]);
    PC_CUDA(cudaGetLastError());
    P->launches++;
  }
  ncclResult_t gr = g_nccl.GroupStart();
  if (gr != ncclSuccess) return nccl_fail(gr, "ncclGroupStart");
  for (size_t i = 0; i < owned.size() && gr == ncclSuccess; i++)
    gr = g_nccl.Send(P->d_recv.get() + off[i], owned[i].rows.size() * dof, ncclDouble, owned[i].rank, comm, P->stream);
  for (size_t i = 0; i < ghost.size() && gr == ncclSuccess; i++)
    gr = g_nccl.Recv(U_loc + (size_t)ghost[i].first_row * dof, (size_t)ghost[i].nrows * dof, ncclDouble, ghost[i].rank, comm, P->stream);
  ncclResult_t ge = g_nccl.GroupEnd();
  if (gr != ncclSuccess) return nccl_fail(gr, "ncclSend/ncclRecv (state halo)");
  if (ge != ncclSuccess) return nccl_fail(ge, "ncclGroupEnd");
  P->launches++;
  return 0;
}

}  // namespace pc

extern "C" {

int petiga_cuda_comm_unique_id(void* id128) {
  if (!id128) return PETIGA_CUDA_ERR_ARG;
  int rc = pc::nccl_load();
  if (rc) return rc;
  ncclUniqueId id;
  ncclResult_t r = pc::g_nccl.GetUniqueId(&id);
  if (r != ncclSuccess) return pc::nccl_fail(r, "ncclGetUniqueId");
  static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is 128 bytes");
  memcpy(id128, &id, 128);
  return 0;
}

int petiga_cuda_comm_init(void** nccl_comm, int nranks, int rank, const void* id128, int device) {
  if (!nccl_comm || !id128) return PETIGA_CUDA_ERR_ARG;
  int rc = pc::nccl_load();
  if (rc) return rc;
  PC_CUDA(cudaSetDevice(device));
  ncclUniqueId id;
  memcpy(&id, id128, 128);
  ncclComm_t comm = nullptr;
  ncclResult_t r = pc::g_nccl.CommInitRank(&comm, nranks, id, rank);
  if (r != ncclSuccess) return pc::nccl_fail(r, "ncclCommInitRank");
  *nccl_comm = comm;
  return 0;
}

int petiga_cuda_comm_destroy(void* nccl_comm) {
  if (!nccl_comm) return 0;
  int rc = pc::nccl_load();
  if (rc) return rc;
  ncclResult_t r = pc::g_nccl.CommDestroy((ncclComm_t)nccl_comm);
  if (r != ncclSuccess) return pc::nccl_fail(r, "ncclCommDestroy");
  return 0;
}

}  // extern "C"
