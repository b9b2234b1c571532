// api.cu -- the C ABI of libckm.so (include/ckm.h): engine lifecycle, model and sequence databases.
// The search itself is in search.cu, the reduction in reduce.cu.
#include <algorithm>
#include <cmath>
#include <cstring>
#include <fstream>
#include <numeric>
#include <stdexcept>
#include <atomic>
#include "engine.hpp"
#include "pool.hpp"

namespace ckm {
const std::string &get_error();
int models_build_device(ckm_models &db);
void models_free_device(ckm_models &db);
}  // namespace ckm

using namespace ckm;

namespace ckm { extern std::atomic<int> g_live_engines; }

extern "C" {

const char *ckm_last_error(void) { return get_error().c_str(); }
const char *ckm_version(void) { return "checkm_b200 0.1 (sm_100a)"; }

int ckm_init(int device, ckm_engine **out) {
  if (!out) { set_error("ckm_init: null output"); return CKM_EINVAL; }
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) {
    set_error("no CUDA device: libckm.so has no CPU fallback (cudaGetDeviceCount: " + std::string(cudaGetErrorString(e)) + ")");
    return CKM_ENODEVICE;
  }
  if (device < 0 || device >= ndev) { set_error("ckm_init: device index out of range"); return CKM_EINVAL; }
  CKM_CUDA(cudaSetDevice(device));
  ckm_engine *eng = new ckm_engine();
  eng->device = device;
  CKM_CUDA(cudaGetDeviceProperties(&eng->prop, device));
  if (eng->prop.major < 10) {
    set_error("libckm.so is built for sm_100a (B200); found compute capability " + std::to_string(eng->prop.major) + "." + std::to_string(eng->prop.minor));
    delete eng;
    return CKM_ENODEVICE;
  }
  CKM_CUDA(cudaStreamCreateWithFlags(&eng->stream, cudaStreamNonBlocking));
  for (auto &ev : eng->ev) CKM_CUDA(cudaEventCreate(&ev));
  // the class streams carry the latency-bound domain-definition kernels: highest priority, so that their few blocks
  // are placed ahead of the throughput kernels of another engine sharing the device
  int prio_lo = 0, prio_hi = 0;
  CKM_CUDA(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
  for (auto &s : eng->cls) CKM_CUDA(cudaStreamCreateWithPriority(&s, cudaStreamNonBlocking, prio_hi));
  CKM_CUDA(cudaStreamCreateWithPriority(&eng->aux, cudaStreamNonBlocking, prio_hi));
  for (auto &ev : eng->cls_ev) CKM_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
  CKM_CUDA(cudaEventCreateWithFlags(&eng->fan_ev, cudaEventDisableTiming));
  CKM_CUDA(cudaMalloc((void **)&eng->d_counters, 64 * sizeof(int32_t) + 64));
  {
    // sequence databases come from the device's stream-ordered pool; keep freed blocks cached for the next batch
    cudaMemPool_t mp;
    if (cudaDeviceGetDefaultMemPool(&mp, device) == cudaSuccess) { uint64_t keep = ~0ull; cudaMemPoolSetAttribute(mp, cudaMemPoolAttrReleaseThreshold, &keep); }
  }
  std::memset(&eng->stats, 0, sizeof(eng->stats));
  ckm::g_live_engines.fetch_add(1);
  *out = eng;
  return CKM_OK;
}

void ckm_destroy(ckm_engine *e) {
  if (!e) return;
  ckm::g_live_engines.fetch_sub(1);
  cudaSetDevice(e->device);
  cudaStreamSynchronize(e->stream);
  for (auto &ev : e->ev) cudaEventDestroy(ev);
  for (auto &s : e->cls) { cudaStreamSynchronize(s); cudaStreamDestroy(s); }
  if (e->aux) { cudaStreamSynchronize(e->aux); cudaStreamDestroy(e->aux); }
  for (auto &ev : e->cls_ev) cudaEventDestroy(ev);
  cudaEventDestroy(e->fan_ev);
  cudaFree(e->d_counters);
  workspace_release(e);
  cudaStreamDestroy(e->stream);
  delete e;
}

int ckm_device_name(ckm_engine *e, char *buf, int buflen) {
  if (!e || !buf || buflen <= 0) { set_error("ckm_device_name: bad argument"); return CKM_EINVAL; }
  std::snprintf(buf, (size_t)buflen, "%s (sm_%d%d, %d SMs)", e->prop.name, e->prop.major, e->prop.minor, e->prop.multiProcessorCount);
  return CKM_OK;
}

// ---------------------------------------------------------------------------------------------
// models
// ---------------------------------------------------------------------------------------------
int ckm_models_load(ckm_engine *e, const char *hmm_path, ckm_models **out) {
  if (!e || !hmm_path || !out) { set_error("ckm_models_load: bad argument"); return CKM_EINVAL; }
  ckm_models *db = new ckm_models();
  db->engine = e;
  try {
    db->models = read_hmm_file(hmm_path);
  } catch (const std::exception &ex) {
    set_error(ex.what());
    delete db;
    std::ifstream probe(hmm_path);
    return probe ? CKM_EFORMAT : CKM_EIO;
  }
  cudaSetDevice(e->device);
  int st = models_build_device(*db);
  if (st != CKM_OK) { models_free_device(*db); delete db; return st; }
  *out = db;
  return CKM_OK;
}

int ckm_models_count(const ckm_models *m) { return m ? (int)m->models.size() : 0; }

int ckm_models_info(const ckm_models *m, int idx, ckm_model_info *out) {
  if (!m || !out || idx < 0 || idx >= (int)m->models.size()) { set_error("ckm_models_info: bad argument"); return CKM_EINVAL; }
  const Model &md = m->models[idx];
  std::memset(out, 0, sizeof(*out));
  std::strncpy(out->name, md.name.c_str(), sizeof(out->name) - 1);
  std::strncpy(out->acc, md.acc.c_str(), sizeof(out->acc) - 1);
  std::strncpy(out->desc, md.desc.c_str(), sizeof(out->desc) - 1);
  out->M = md.M;
  out->has_ga = md.has_ga; out->has_tc = md.has_tc; out->has_nc = md.has_nc;
  for (int z = 0; z < 2; ++z) { out->ga[z] = md.ga[z]; out->tc[z] = md.tc[z]; out->nc[z] = md.nc[z]; out->ga_d[z] = md.ga_d[z]; out->tc_d[z] = md.tc_d[z]; out->nc_d[z] = md.nc_d[z]; }
  for (int z = 0; z < 6; ++z) out->evparam[z] = md.evparam[z];
  return CKM_OK;
}

int ckm_models_find(const ckm_models *m, const char *key) {
  if (!m || !key) return -1;
  for (size_t i = 0; i < m->models.size(); ++i)
    if (m->models[i].acc == key || m->models[i].name == key) return (int)i;
  return -1;
}

int ckm_models_select(const ckm_models *m, const char *const *keys, int nkeys, int32_t *idx_out, int *n_out) {
  if (!m || !keys || !idx_out || !n_out || nkeys < 0) { set_error("ckm_models_select: bad argument"); return CKM_EINVAL; }
  std::vector<char> want(m->models.size(), 0);
  for (int i = 0; i < nkeys; ++i) {
    int idx = ckm_models_find(m, keys[i]);
    if (idx < 0) { set_error(std::string("ckm_models_select: key not in database: ") + keys[i]); return CKM_ENOTFOUND; }
    want[idx] = 1;
  }
  int n = 0;
  for (size_t i = 0; i < want.size(); ++i) if (want[i]) idx_out[n++] = (int32_t)i;   // database order, like hmmfetch -f on an indexed file
  *n_out = n;
  return CKM_OK;
}

int ckm_models_write(const ckm_models *m, const int32_t *idx, int n, const char *out_path) {
  if (!m || !out_path || (n > 0 && !idx)) { set_error("ckm_models_write: bad argument"); return CKM_EINVAL; }
  std::ofstream out(out_path);
  if (!out) { set_error(std::string("cannot write ") + out_path); return CKM_EIO; }
  for (int i = 0; i < n; ++i) {
    if (idx[i] < 0 || idx[i] >= (int)m->models.size()) { set_error("ckm_models_write: index out of range"); return CKM_EINVAL; }
    out << m->models[idx[i]].text;
  }
  return out.good() ? CKM_OK : CKM_EIO;
}

void ckm_models_free(ckm_models *m) {
  if (!m) return;
  if (m->engine) cudaSetDevice(m->engine->device);
  models_free_device(*m);
  delete m;
}

// ---------------------------------------------------------------------------------------------
// sequences
// ---------------------------------------------------------------------------------------------
int ckm_digitize(const char *text, int64_t n, uint8_t *out) {
  if ((!text || !out) && n > 0) { set_error("ckm_digitize: bad argument"); return CKM_EINVAL; }
  for (int64_t i = 0; i < n; ++i) {
    int c = digitize_char((unsigned char)text[i]);
    out[i] = (uint8_t)(c < 0 ? 26 : c);       // unknown symbols become X
  }
  return CKM_OK;
}

// FASTA text -> digitised residues + CSR offsets + the header lines (text after '>', joined by '\n').  A header line starts
// with '>' at the beginning of a line; whitespace inside sequence lines is dropped; bytes before the first header are ignored.
int ckm_fasta_parse(const char *text, int64_t n, uint8_t *residues_out, int64_t *offsets_out, int32_t max_records,
                    char *headers_out, int64_t headers_cap, int32_t *nrec_out, int64_t *nres_out, int64_t *hdr_bytes_out) {
  if ((!text && n > 0) || !residues_out || !offsets_out || !headers_out || !nrec_out || !nres_out || !hdr_bytes_out) { set_error("ckm_fasta_parse: bad argument"); return CKM_EINVAL; }
  static uint8_t lut[256]; static bool lut_ready = false;
  if (!lut_ready) {
    for (int c = 0; c < 256; ++c) {
      const bool ws = (c == ' ' || (c >= 9 && c <= 13));
      const int d = digitize_char((unsigned char)c);
      lut[c] = ws ? 255 : (uint8_t)(d < 0 ? 26 : d);      // 255 = skip; unknown symbols become X like ckm_digitize
    }
    lut_ready = true;
  }
  int32_t nrec = 0; int64_t nres = 0, hb = 0, i = 0;
  bool started = false;
  while (i < n) {
    const char *nlp = (const char *)std::memchr(text + i, '\n', (size_t)(n - i));
    const int64_t e = nlp ? (nlp - text) : n;                  // line is [i, e)
    if (text[i] == '>') {
      if (nrec >= max_records) { set_error("ckm_fasta_parse: more records than the caller allowed for"); return CKM_ECAPACITY; }
      int64_t he = e;
      if (he > i + 1 && text[he - 1] == '\r') --he;
      const int64_t len = he - (i + 1);
      if (hb + len + 1 > headers_cap) { set_error("ckm_fasta_parse: header buffer too small"); return CKM_ECAPACITY; }
      if (nrec > 0) headers_out[hb++] = '\n';
      std::memcpy(headers_out + hb, text + i + 1, (size_t)len); hb += len;
      offsets_out[nrec++] = nres;
      started = true;
    } else if (started) {
      for (int64_t j = i; j < e; ++j) { const uint8_t c = lut[(unsigned char)text[j]]; if (c != 255) residues_out[nres++] = c; }
    }
    i = e + 1;
  }
  offsets_out[nrec] = nres;
  *nrec_out = nrec; *nres_out = nres; *hdr_bytes_out = hb;
  return CKM_OK;
}

static inline uint8_t unbiased_byteify_h(float scale_b, float sc) {
  sc = -1.0f * roundf(scale_b * sc);
  return (sc > 255.0f) ? 255 : (uint8_t)sc;
}
static inline int16_t wordify_h(float scale_w, float sc) {
  sc = roundf(scale_w * sc);
  if (sc >= 32767.0f) return 32767;
  if (sc <= -32768.0f) return -32768;
  return (int16_t)sc;
}

int ckm_seqdb_create(ckm_engine *e, const uint8_t *residues, const int64_t *seq_offsets, int32_t nseq,
                     const int32_t *bin_of_seq, int32_t nbins, ckm_seqdb **out) {
  if (!e || !out || nseq < 0 || (nseq > 0 && (!residues || !seq_offsets))) { set_error("ckm_seqdb_create: bad argument"); return CKM_EINVAL; }
  if (nbins < 1) nbins = 1;
  cudaSetDevice(e->device);
  ckm_seqdb *db = new ckm_seqdb();
  db->engine = e; db->nseq = nseq; db->nbins = nbins;
  db->offsets.assign(seq_offsets, seq_offsets + nseq + 1);
  db->bin_of_seq.assign(nseq, 0);
  if (bin_of_seq) db->bin_of_seq.assign(bin_of_seq, bin_of_seq + nseq);
  db->bin_nseq.assign(nbins, 0); db->bin_first_seq.assign(nbins, 0);
  db->len.resize(nseq);
  std::vector<int64_t> poff(nseq + 1, 0);
  const float scale_b = (float)(3.0 / 0.69314718055994529), scale_w = (float)(500.0 / 0.69314718055994529);
  std::vector<float> nullsc(nseq), msvB(nseq), lenA(nseq), lenB(nseq);
  std::vector<int32_t> tjb(nseq);
  std::vector<int16_t> tmove(nseq);
  int64_t pos = 0;
  for (int s = 0; s < nseq; ++s) {
    int64_t L = seq_offsets[s + 1] - seq_offsets[s];
    if (L < 0 || L > 100000000) { set_error("ckm_seqdb_create: bad sequence offsets"); delete db; return CKM_EINVAL; }
    int b = db->bin_of_seq[s];
    if (b < 0 || b >= nbins) { set_error("ckm_seqdb_create: bin index out of range"); delete db; return CKM_EINVAL; }
    if (db->bin_nseq[b] == 0) db->bin_first_seq[b] = s;
    else if (db->bin_first_seq[b] + db->bin_nseq[b] != s) { set_error("ckm_seqdb_create: sequences of a bin must be contiguous"); delete db; return CKM_EINVAL; }
    db->bin_nseq[b]++;
    db->len[s] = (int32_t)L;
    db->maxL = std::max(db->maxL, (int32_t)L);
    poff[s] = pos;
    pos += (L + 15) / 16 * 16;
    // per-sequence length model (SURVEY.md A.4/A.5): null1 score, MSV move cost, Viterbi move score
    float p1 = (float)L / (float)(L + 1);
    lenA[s] = (float)L * logf(p1); lenB[s] = logf(1.0f - p1);
    nullsc[s] = (float)L * logf(p1) + logf(1.0f - p1);
    tjb[s] = unbiased_byteify_h(scale_b, logf(3.0f / (float)(L + 3)));
    tmove[s] = wordify_h(scale_w, logf(3.0f / (float)(L + 3)));
    msvB[s] = 2.0f * (float)tjb[s] + scale_b * (3.0f + nullsc[s]);
  }
  poff[nseq] = pos;
  db->nres = seq_offsets[nseq] - seq_offsets[0];
  db->padded_bytes = pos + 16;
  std::vector<uint8_t> padded((size_t)db->padded_bytes, (uint8_t)CODE_PAD);
  for (int s = 0; s < nseq; ++s) {
    const uint8_t *src = residues + seq_offsets[s];
    uint8_t *dst = padded.data() + poff[s];
    for (int32_t i = 0; i < db->len[s]; ++i) dst[i] = src[i] < KP ? src[i] : (uint8_t)26;
  }
  std::vector<int32_t> order(nseq);
  std::iota(order.begin(), order.end(), 0);
  std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return db->len[a] > db->len[b]; });
  auto up = [&](void **d, const void *h, size_t bytes) -> int {
    CKM_CUDA(cudaMallocAsync(d, std::max<size_t>(bytes, 16), e->stream));     // stream-ordered: no device-wide synchronisation
    if (bytes) CKM_CUDA(cudaMemcpyAsync(*d, h, bytes, cudaMemcpyHostToDevice, e->stream));
    return CKM_OK;
  };
  int st = CKM_OK;
  if (!st) st = up((void **)&db->d_res, padded.data(), padded.size());
  if (!st) st = up((void **)&db->d_off, poff.data(), poff.size() * sizeof(int64_t));
  if (!st) st = up((void **)&db->d_len, db->len.data(), (size_t)nseq * sizeof(int32_t));
  if (!st) st = up((void **)&db->d_bin, db->bin_of_seq.data(), (size_t)nseq * sizeof(int32_t));
  if (!st) st = up((void **)&db->d_nullsc, nullsc.data(), (size_t)nseq * sizeof(float));
  if (!st) st = up((void **)&db->d_tjb, tjb.data(), (size_t)nseq * sizeof(int32_t));
  if (!st) st = up((void **)&db->d_msvB, msvB.data(), (size_t)nseq * sizeof(float));
  if (!st) st = up((void **)&db->d_lenA, lenA.data(), (size_t)nseq * sizeof(float));
  if (!st) st = up((void **)&db->d_lenB, lenB.data(), (size_t)nseq * sizeof(float));
  if (!st) st = up((void **)&db->d_tmove_w, tmove.data(), (size_t)nseq * sizeof(int16_t));
  if (!st) st = up((void **)&db->d_order, order.data(), (size_t)nseq * sizeof(int32_t));
  if (!st) st = up((void **)&db->d_bin_nseq, db->bin_nseq.data(), (size_t)nbins * sizeof(int32_t));
  if (!st) { cudaError_t ce = cudaStreamSynchronize(e->stream); if (ce != cudaSuccess) st = cuda_fail(ce, "seqdb upload"); }
  if (st) { ckm_seqdb_free(db); return st; }
  *out = db;
  return CKM_OK;
}

void ckm_seqdb_free(ckm_seqdb *db) {
  if (!db) return;
  if (db->engine) {
    cudaSetDevice(db->engine->device);
    cudaStream_t st = db->engine->stream;
    void *ptrs[] = {db->d_res, db->d_off, db->d_len, db->d_bin, db->d_nullsc, db->d_tjb, db->d_msvB, db->d_lenA, db->d_lenB, db->d_tmove_w, db->d_order, db->d_bin_nseq};
    for (void *q : ptrs) if (q) cudaFreeAsync(q, st);
  }
  delete db;
}

void ckm_free(void *p) { std::free(p); }
void ckm_hits_free(ckm_hit *hits) { std::free(hits); }

int ckm_last_stats(const ckm_engine *e, ckm_stats *out) {
  if (!e || !out) { set_error("ckm_last_stats: bad argument"); return CKM_EINVAL; }
  *out = e->stats;
  return CKM_OK;
}

int ckm_workspace_bytes(const ckm_engine *e, int64_t *bytes_out) {
  if (!e || !bytes_out) { set_error("ckm_workspace_bytes: bad argument"); return CKM_EINVAL; }
  *bytes_out = 0;
  for (const auto &w : e->ws) *bytes_out += (int64_t)w.bytes;
  return CKM_OK;
}

}  // extern "C"
