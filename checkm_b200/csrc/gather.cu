// gather.cu -- multi-GPU: the per-bin QA rows of all ranks on every rank, one NCCL all-gather over NVLink (BASELINE.json
// configs[3]: "NCCL gather of qa table"; SURVEY.md 8e).  Bins are independent, so this is the only inter-GPU traffic of a run.
// libnccl is bound at run time (dlopen): a single-GPU process never needs it, and a torch process has it loaded already.
#include <dlfcn.h>
#include <cstring>
#include <mutex>
#include <vector>
#include "engine.hpp"
#include "pool.hpp"

using namespace ckm;

namespace {

typedef struct { char internal[128]; } nccl_uid;
typedef int (*fn_get_uid)(nccl_uid *);
typedef int (*fn_comm_init)(void **, int, nccl_uid, int);
typedef int (*fn_all_gather)(const void *, void *, size_t, int, void *, cudaStream_t);
typedef int (*fn_comm_destroy)(void *);
typedef const char *(*fn_err)(int);

struct Nccl {
  void *h = nullptr;
  fn_get_uid get_uid = nullptr; fn_comm_init comm_init = nullptr; fn_all_gather all_gather = nullptr; fn_comm_destroy comm_destroy = nullptr; fn_err err = nullptr;
};

int load_nccl(Nccl **out) {
  static Nccl lib; static std::once_flag once; static bool ok = false;
  std::call_once(once, [] {
    for (const char *name : {"libnccl.so.2", "libnccl.so"}) { lib.h = dlopen(name, RTLD_NOW | RTLD_GLOBAL); if (lib.h) break; }
    if (!lib.h) return;
    lib.get_uid = (fn_get_uid)dlsym(lib.h, "ncclGetUniqueId");
    lib.comm_init = (fn_comm_init)dlsym(lib.h, "ncclCommInitRank");
    lib.all_gather = (fn_all_gather)dlsym(lib.h, "ncclAllGather");
    lib.comm_destroy = (fn_comm_destroy)dlsym(lib.h, "ncclCommDestroy");
    lib.err = (fn_err)dlsym(lib.h, "ncclGetErrorString");
    ok = lib.get_uid && lib.comm_init && lib.all_gather && lib.comm_destroy;
  });
  if (!ok) { set_error("NCCL is not available (libnccl.so.2 could not be loaded)"); return CKM_ENODEVICE; }
  *out = &lib;
  return CKM_OK;
}

int nccl_fail(Nccl *n, int rc, const char *what) {
  set_error(std::string("NCCL error in ") + what + ": " + (n->err ? n->err(rc) : "?"));
  return CKM_ECUDA;
}

}  // namespace

extern "C" {

int ckm_nccl_unique_id(uint8_t *id_out, int32_t nbytes) {
  if (!id_out || nbytes < 128) { set_error("ckm_nccl_unique_id: need a 128-byte buffer"); return CKM_EINVAL; }
  Nccl *n; int rc;
  if ((rc = load_nccl(&n))) return rc;
  nccl_uid uid;
  if ((rc = n->get_uid(&uid))) return nccl_fail(n, rc, "ncclGetUniqueId");
  std::memcpy(id_out, uid.internal, 128);
  return CKM_OK;
}

int ckm_nccl_comm_init(ckm_engine *e, int32_t world, int32_t rank, const uint8_t *id, void **comm_out) {
  if (!e || !id || !comm_out || world < 1 || rank < 0 || rank >= world) { set_error("ckm_nccl_comm_init: bad argument"); return CKM_EINVAL; }
  Nccl *n; int rc;
  if ((rc = load_nccl(&n))) return rc;
  CKM_CUDA(cudaSetDevice(e->device));
  nccl_uid uid;
  std::memcpy(uid.internal, id, 128);
  void *comm = nullptr;
  if ((rc = n->comm_init(&comm, world, uid, rank))) return nccl_fail(n, rc, "ncclCommInitRank");
  *comm_out = comm;
  return CKM_OK;
}

void ckm_nccl_comm_destroy(void *comm) {
  Nccl *n;
  if (comm && load_nccl(&n) == CKM_OK) n->comm_destroy(comm);
}

// Every rank contributes nrows (<= nrows_max) rows; rows_out receives world * nrows_max rows (rank r's rows start at
// r * nrows_max), counts_out the row count of every rank.  One ncclAllGather of world x (8 + nrows_max * sizeof(row)) bytes.
int ckm_allgather_qa(ckm_engine *e, void *nccl_comm, const ckm_qa_row *rows, int32_t nrows, int32_t nrows_max,
                     int32_t world, ckm_qa_row *rows_out, int32_t *counts_out) {
  if (!e || !nccl_comm || (!rows && nrows > 0) || !rows_out || !counts_out || nrows < 0 || nrows > nrows_max || world < 1) {
    set_error("ckm_allgather_qa: bad argument"); return CKM_EINVAL;
  }
  Nccl *n; int rc;
  if ((rc = load_nccl(&n))) return rc;
  CKM_CUDA(cudaSetDevice(e->device));
  const size_t slot = 8 + (size_t)nrows_max * sizeof(ckm_qa_row);
  const size_t need = slot * ((size_t)world + 1);
  uint8_t *d_send;
  if ((rc = workspace(e, Ws::Gather, need, &d_send))) return rc;
  uint8_t *d_recv = d_send + slot;
  std::vector<uint8_t> host(slot * (size_t)world, 0);
  const int64_t cnt = nrows;
  std::memcpy(host.data(), &cnt, 8);
  if (nrows) std::memcpy(host.data() + 8, rows, (size_t)nrows * sizeof(ckm_qa_row));
  CKM_CUDA(cudaMemcpyAsync(d_send, host.data(), slot, cudaMemcpyHostToDevice, e->stream));
  if ((rc = n->all_gather(d_send, d_recv, slot, 0 /* ncclChar */, nccl_comm, e->stream))) return nccl_fail(n, rc, "ncclAllGather");
  CKM_CUDA(cudaMemcpyAsync(host.data(), d_recv, slot * (size_t)world, cudaMemcpyDeviceToHost, e->stream));
  CKM_CUDA(cudaStreamSynchronize(e->stream));
  for (int r = 0; r < world; ++r) {
    int64_t c;
    std::memcpy(&c, host.data() + slot * r, 8);
    if (c < 0 || c > nrows_max) { set_error("ckm_allgather_qa: corrupt row count from a peer"); return CKM_EINVAL; }
    counts_out[r] = (int32_t)c;
    std::memcpy(rows_out + (size_t)r * nrows_max, host.data() + slot * r + 8, (size_t)c * sizeof(ckm_qa_row));
  }
  return CKM_OK;
}

}  // extern "C"
