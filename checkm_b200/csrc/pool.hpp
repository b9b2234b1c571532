// pool.hpp -- the engine's workspace table: one grow-only device buffer per role (ckm::Ws), reused by every later call
#pragma once
#include <algorithm>
#include "engine.hpp"

namespace ckm {

// The engine's buffer for `key`, at least `bytes` (and 256) long.  A buffer that is too small is freed and allocated again with
// 25% slack, or exactly `bytes` when the slack does not fit; its contents are not kept.
template <class T> int workspace(ckm_engine *e, Ws key, size_t bytes, T **out) {
  auto &w = e->ws[(int)key];
  bytes = std::max<size_t>(bytes, 256);
  if (w.bytes < bytes) {
    cudaFree(w.p);
    w.p = nullptr; w.bytes = 0;
    const size_t want = bytes + bytes / 4;
    if (cudaMalloc(&w.p, want) == cudaSuccess) w.bytes = want;
    else {
      const cudaError_t err = cudaMalloc(&w.p, bytes);
      if (err != cudaSuccess) { w.p = nullptr; *out = nullptr; return cuda_fail(err, "cudaMalloc(workspace)"); }
      w.bytes = bytes;
    }
  }
  *out = static_cast<T *>(w.p);
  return CKM_OK;
}

// Frees every workspace (the next call allocates what it needs again).  No stream of the engine may still use them.
inline void workspace_release(ckm_engine *e) {
  for (auto &w : e->ws) { cudaFree(w.p); w.p = nullptr; w.bytes = 0; }
}

}  // namespace ckm
