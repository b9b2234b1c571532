// search.cu -- the search driver: launches the filter cascade and the domain-definition stages on the engine's
// stream and assembles the hit table.  Replaces the body of `hmmsearch` behind checkm/hmmer.py:61-74.
#include <algorithm>
#include <atomic>
#include <chrono>
#include <cstdio>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <vector>
#include "engine.hpp"
#include "stages.hpp"
#include "pool.hpp"

using namespace ckm;

namespace ckm {

std::atomic<int> g_live_engines{0};     // engines alive in this process: they share the envelope-scratch budget

static bool use_blocked_kernels();
static bool use_packed_viterbi() { const char *v = std::getenv("CKM_VITP"); return use_blocked_kernels() && !(v != nullptr && v[0] == '0'); }
static int fan_out(ckm_engine *e);
static int fan_in(ckm_engine *e);
enum { CTR_UNIT4 = 0, CTR_UNIT8, CTR_UNIT16, CTR_UNIT32, CTR_CAND, CTR_MSV, CTR_BIAS, CTR_VIT, CTR_FWD, CTR_ENV, CTR_DOM, CTR_VREDO, CTR_SSVRES, CTR_VWORK = 16 /* .. 25: cursors of the packed-Viterbi class kernels */, CTR_N = 32 };

struct ActiveMasks {
  int32_t *model_slot = nullptr;
  uint8_t *tile_active = nullptr, *model_active = nullptr;    // nullptr: every model is queried in every bin
};

// Builds the per-bin activity masks for a query subset.  bin_model_offsets == nullptr: the same nmodels queries for all bins.
static int build_masks(ckm_engine *e, const ckm_models *m, const ckm_seqdb *db, const int32_t *model_idx, int32_t nmodels,
                       const int64_t *bin_model_offsets, ActiveMasks &am, std::vector<int32_t> &slot_of_model) {
  cudaStream_t st = e->stream;
  const int ndb = (int)m->models.size(), nbins = db->nbins, ntiles = (int)m->tiles.size();
  slot_of_model.assign(ndb, -1);
  bool all = (bin_model_offsets == nullptr) && (model_idx == nullptr || nmodels == ndb);
  if (model_idx == nullptr) { for (int i = 0; i < ndb; ++i) slot_of_model[i] = i; }
  else if (bin_model_offsets == nullptr) {
    for (int i = 0; i < nmodels; ++i) {
      if (model_idx[i] < 0 || model_idx[i] >= ndb) { set_error("model index out of range"); return CKM_EINVAL; }
      if (slot_of_model[model_idx[i]] >= 0) { set_error("duplicate model index in query list"); return CKM_EINVAL; }
      slot_of_model[model_idx[i]] = i;
    }
    if (all) for (int i = 0; i < ndb; ++i) if (slot_of_model[i] < 0) all = false;
  }
  int rc;
  if ((rc = workspace(e, Ws::ModelSlot, sizeof(int32_t) * ndb, &am.model_slot))) return rc;
  CKM_CUDA(cudaMemcpyAsync(am.model_slot, slot_of_model.data(), sizeof(int32_t) * ndb, cudaMemcpyHostToDevice, st));
  if (all) return CKM_OK;
  std::vector<uint8_t> ma((size_t)nbins * ndb, 0), ta((size_t)nbins * ntiles, 0);
  for (int b = 0; b < nbins; ++b) {
    if (bin_model_offsets == nullptr) {
      for (int i = 0; i < nmodels; ++i) ma[(size_t)b * ndb + model_idx[i]] = 1;
    } else {
      for (int64_t i = bin_model_offsets[b]; i < bin_model_offsets[b + 1]; ++i) {
        if (model_idx[i] < 0 || model_idx[i] >= ndb) { set_error("model index out of range"); return CKM_EINVAL; }
        ma[(size_t)b * ndb + model_idx[i]] = 1;
      }
    }
    for (int t = 0; t < ntiles; ++t) {
      const TileDesc &td = m->tiles[t];
      uint8_t any = 0;
      for (int j = 0; j < td.nmodels; ++j) any |= ma[(size_t)b * ndb + m->tile_models[td.first_model + j].model];
      ta[(size_t)b * ntiles + t] = any;
    }
    // a chained model is addressed through its first tile
  }
  if ((rc = workspace(e, Ws::ModelActive, ma.size(), &am.model_active))) return rc;
  if ((rc = workspace(e, Ws::TileActive, ta.size(), &am.tile_active))) return rc;
  CKM_CUDA(cudaMemcpyAsync(am.model_active, ma.data(), ma.size(), cudaMemcpyHostToDevice, st));
  CKM_CUDA(cudaMemcpyAsync(am.tile_active, ta.data(), ta.size(), cudaMemcpyHostToDevice, st));
  CKM_CUDA(cudaStreamSynchronize(st));     // host vectors go out of scope
  return CKM_OK;
}

// Stage 1: SSV pre-filter over all pairs -> candidate list; exact MSV on the candidates -> pass list.
struct Stage1 {
  int2 *cand = nullptr; Candidate *pass = nullptr; unsigned long long *cells = nullptr;
  int32_t cand_cap = 0, pass_cap = 0;
};

// Queue capacities: a fraction of the pairs (SSV forwards ~3%, exact MSV keeps ~2%; 1/6 and 1/12 leave a wide margin), all in
// 64-bit arithmetic, never beyond QUEUE_MAX entries.  `attempt` > 0 is a retry after an overflow: the fractions grow 8-fold
// each time, so the third attempt holds every pair (or QUEUE_MAX of them).
constexpr int64_t QUEUE_MAX = (int64_t)1 << 30;
static int32_t queue_cap(int64_t n_pairs, int64_t divisor, int attempt) {
  int64_t want = n_pairs / divisor + 65536;
  for (int a = 0; a < attempt && want < n_pairs; ++a) want *= 8;
  return (int32_t)std::min<int64_t>(std::min<int64_t>(n_pairs, QUEUE_MAX), std::max<int64_t>((int64_t)1 << 16, want));
}

static int run_stage1(ckm_engine *e, const ckm_models *m, const ckm_seqdb *db, ActiveMasks &am, int64_t n_pairs,
                      Stage1 &s1, int32_t *xj_dense, int attempt = 0) {
  cudaStream_t st = e->stream;
  int rc;
  s1.cand_cap = queue_cap(n_pairs, 6, attempt);
  const int64_t n_bypass = (int64_t)m->ssv_bypass.size() * db->nseq;          // models without SSV tiles: every pair is a candidate
  s1.cand_cap = (int32_t)std::min<int64_t>(QUEUE_MAX, (int64_t)s1.cand_cap + n_bypass);
  s1.pass_cap = queue_cap(n_pairs, 12, attempt);
  if ((rc = workspace(e, Ws::Cand, sizeof(int2) * (size_t)s1.cand_cap, &s1.cand))) return rc;
  if ((rc = workspace(e, Ws::Pass, sizeof(Candidate) * (size_t)s1.pass_cap, &s1.pass))) return rc;
  if ((rc = workspace(e, Ws::Cells, sizeof(unsigned long long), &s1.cells))) return rc;
  CKM_CUDA(cudaMemsetAsync(e->d_counters, 0, CTR_N * sizeof(int32_t), st));
  CKM_CUDA(cudaMemsetAsync(s1.cells, 0, sizeof(unsigned long long), st));
  const int nsm = e->prop.multiProcessorCount;
  bool need_bnd = false;
  for (int nt : m->chain_ntiles) need_bnd |= (nt > 1);
  const int64_t bnd_stride = ((int64_t)db->maxL + 31) / 16 * 16;
  int16_t *bnd = nullptr;
  if (need_bnd) { if ((rc = workspace(e, Ws::Bnd, (size_t)nsm * SSV_WARPS_HOST * 2 * bnd_stride * sizeof(int16_t), &bnd))) return rc; }
  // group lists per J
  std::vector<int32_t> gl[4];
  for (size_t g = 0; g < m->groups.size(); ++g) gl[m->groups[g].J == 4 ? 0 : (m->groups[g].J == 8 ? 1 : (m->groups[g].J == 16 ? 2 : 3))].push_back((int32_t)g);
  std::vector<int32_t> flat;
  size_t goff[4];
  for (int c = 0; c < 4; ++c) { goff[c] = flat.size(); flat.insert(flat.end(), gl[c].begin(), gl[c].end()); }
  int32_t *glist;
  if ((rc = workspace(e, Ws::GroupList, sizeof(int32_t) * std::max<size_t>(flat.size(), 1), &glist))) return rc;
  if (!flat.empty()) CKM_CUDA(cudaMemcpyAsync(glist, flat.data(), sizeof(int32_t) * flat.size(), cudaMemcpyHostToDevice, st));
  CKM_CUDA(cudaStreamSynchronize(st));

  CKM_CUDA(cudaEventRecord(e->ev[0], st));
  const int Js[4] = {4, 8, 16, 32};
  for (int c = 0; c < 4; ++c) {
    if (gl[c].empty() || db->nseq == 0) continue;
    SsvParams p{};
    p.res = db->d_res; p.off = db->d_off; p.len = db->d_len; p.bin = db->d_bin;
    p.msvB = db->d_msvB; p.tjb = db->d_tjb; p.order = db->d_order;
    p.nseq = db->nseq;
    p.seq_chunk = 128;
    p.nchunks = (db->nseq + p.seq_chunk - 1) / p.seq_chunk;
    p.groups = m->d_groups; p.group_list = glist + goff[c]; p.ngroups = (int32_t)gl[c].size();
    p.tiles = m->d_tiles; p.tile_models = m->d_tile_models;
    p.chain_first_tile = m->d_chain_first_tile; p.chain_ntiles = m->d_chain_ntiles;
    p.tile_blob = m->d_tile_blob;
    p.tile_active = am.tile_active; p.model_active = am.model_active;
    p.ntiles = (int32_t)m->tiles.size(); p.nmodels = (int32_t)m->models.size();
    p.unit_counter = e->d_counters + CTR_UNIT4 + c;
    p.cand = s1.cand; p.cand_count = e->d_counters + CTR_CAND; p.cand_cap = s1.cand_cap;
    p.bnd = bnd; p.bnd_stride = bnd_stride;
    p.cells = s1.cells;
    { const char *v = std::getenv("CKM_SSV_RESOLVE"); p.resolve = (v != nullptr && v[0] == '0') ? 0 : 1; }
    p.ms = m->d_scalars; p.nullsc = db->d_nullsc;
    p.pass = s1.pass; p.pass_count = e->d_counters + CTR_MSV; p.pass_cap = s1.pass_cap;
    p.resolved_count = e->d_counters + CTR_SSVRES;
    p.xj_dense = xj_dense; p.model_slot = am.model_slot;
    p.F1 = 0.02;
    int64_t maxbytes = 0;
    for (int g : gl[c]) maxbytes = std::max<int64_t>(maxbytes, m->groups[g].table_bytes);
    const int64_t units = (int64_t)p.ngroups * p.nchunks;
    const int grid = (int)std::min<int64_t>(nsm, units);
    if ((rc = launch_ssv(Js[c], m->ssv_tmem, p, grid, (size_t)maxbytes, st))) return rc;
    e->stats.kernel_launches++;
  }
  if (!m->ssv_bypass.empty()) {
    if ((rc = launch_ssv_bypass(m->d_ssv_bypass, (int32_t)m->ssv_bypass.size(), db->nseq, db->d_len, db->d_bin,
                                am.model_active, (int32_t)m->models.size(), s1.cand, e->d_counters + CTR_CAND, s1.cand_cap, st))) return rc;
    e->stats.kernel_launches++;
  }
  CKM_CUDA(cudaEventRecord(e->ev[1], st));
  // exact MSV on the candidates
  {
    MsvParams p{};
    p.res = db->d_res; p.off = db->d_off; p.len = db->d_len; p.nullsc = db->d_nullsc; p.tjb = db->d_tjb;
    p.ms = m->d_scalars; p.rbv = m->d_rbv; p.rmb = m->d_rmb;
    p.cand = s1.cand; p.cand_count = e->d_counters + CTR_CAND; p.cand_cap = s1.cand_cap;
    p.out = s1.pass; p.out_count = e->d_counters + CTR_MSV; p.out_cap = s1.pass_cap;
    p.xj_dense = xj_dense; p.model_slot = am.model_slot; p.nseq = db->nseq;
    p.row_bytes = (m->maxM + 2 + 15) / 16 * 16;
    p.F1 = 0.02;
    p.use_blk = use_blocked_kernels() ? 1 : 0;
    if ((rc = fan_out(e))) return rc;
    if (p.use_blk) { for (int c = 0; c < N_BLK_CLASSES; ++c) if ((rc = launch_msv2(p, c, nsm * 16, e->cls[c]))) return rc; }
    if ((rc = launch_msv_exact(p, nsm * 4, e->cls[N_BLK_CLASSES]))) return rc;
    if ((rc = fan_in(e))) return rc;
    e->stats.kernel_launches += 1 + (p.use_blk ? N_BLK_CLASSES : 0);
  }
  CKM_CUDA(cudaEventRecord(e->ev[2], st));
  return CKM_OK;
}


// Stages 2-4 on the MSV survivors: bias filter -> ViterbiFilter -> ForwardParser.  Lists ping-pong between two buffers.
struct Stage2 {
  Candidate *a = nullptr, *b = nullptr, *redo = nullptr;
  int32_t cap = 0;
  Candidate *fwd_list = nullptr;      // survivors of the Forward filter (points into a or b)
};

static int run_stage2(ckm_engine *e, const ckm_models *m, const ckm_seqdb *db, ActiveMasks &am, Stage1 &s1, Stage2 &s2,
                      float *d_filtersc, float *d_vit, float *d_fwd, uint8_t *d_passed) {
  cudaStream_t st = e->stream;
  int rc;
  s2.cap = s1.pass_cap;
  if ((rc = workspace(e, Ws::ListA, sizeof(Candidate) * (size_t)s2.cap, &s2.a))) return rc;
  if ((rc = workspace(e, Ws::ListB, sizeof(Candidate) * (size_t)s2.cap, &s2.b))) return rc;
  if ((rc = workspace(e, Ws::Redo, sizeof(Candidate) * (size_t)s2.cap, &s2.redo))) return rc;
  const int nsm = e->prop.multiProcessorCount;
  FilterParams p{};
  p.res = db->d_res; p.off = db->d_off; p.len = db->d_len; p.lenA = db->d_lenA; p.lenB = db->d_lenB; p.tmove_w = db->d_tmove_w;
  p.ms = m->d_scalars; p.bias_eo = m->d_bias_eo; p.rwv = m->d_rwv; p.twv = m->d_twv; p.rfv = m->d_rfv; p.tfv = m->d_tfv;
  p.twb = m->d_twb; p.rwb = m->d_rwb; p.tfb = m->d_tfb; p.rfb = m->d_rfb;
  p.twp = m->d_twp; p.rwp = m->d_rwp;
  p.redo = s2.redo; p.redo_count = e->d_counters + CTR_VREDO; p.redo_cap = s2.cap;
  p.row_elems = ((m->maxM + 31) / 32) * 32 + 64;
  p.F1 = 0.02; p.F2 = 1e-3; p.F3 = 1e-5;
  p.use_blk = use_blocked_kernels() ? 1 : 0;
  p.dense_filtersc = d_filtersc; p.dense_vit = d_vit; p.dense_fwd = d_fwd; p.dense_passed = d_passed;
  p.model_slot = am.model_slot; p.nseq = db->nseq;
  // bias: pass list (stage 1) -> a
  p.in = s1.pass; p.in_count = e->d_counters + CTR_MSV; p.in_cap = s1.pass_cap;
  p.out = s2.a; p.out_count = e->d_counters + CTR_BIAS; p.out_cap = s2.cap;
  if ((rc = launch_bias(p, nsm * 8, st))) return rc;
  CKM_CUDA(cudaEventRecord(e->ev[3], st));
  // viterbi: a -> b
  p.in = s2.a; p.in_count = e->d_counters + CTR_BIAS; p.in_cap = s2.cap;
  p.out = s2.b; p.out_count = e->d_counters + CTR_VIT; p.out_cap = s2.cap;
  if (use_packed_viterbi()) {
    // packed int16x2 kernels, one per class; what they cannot score exactly (strong hits near the int16 ceiling, models
    // without a class, pairs outside the safety conditions of kernels_vitp.cu) lands in the redo list ...
    p.vit_work = e->d_counters + CTR_VWORK;      // zeroed with the other counters at the start of the cascade
    if ((rc = fan_out(e))) return rc;
    for (int c = 0; c < N_BLK_CLASSES; ++c) if ((rc = launch_vitp(p, c, nsm * 8, e->cls[c]))) return rc;
    if ((rc = fan_in(e))) return rc;
    // ... which the int32 kernels below then take as their input
    p.in = s2.redo; p.in_count = e->d_counters + CTR_VREDO; p.in_cap = s2.cap;
    e->stats.kernel_launches += N_BLK_CLASSES;
  }
  if ((rc = fan_out(e))) return rc;
  if (p.use_blk) { for (int c = 0; c < N_BLK_CLASSES; ++c) if ((rc = launch_vit2(p, c, nsm * 8, e->cls[c]))) return rc; }   // lane-blocked register kernels, one per class
  if ((rc = launch_vit(p, nsm * 4, e->cls[N_BLK_CLASSES]))) return rc;                                      // models beyond the classes (all models when CKM_BLK=0): shared-memory rows
  if ((rc = fan_in(e))) return rc;
  CKM_CUDA(cudaEventRecord(e->ev[4], st));
  // forward: b -> a
  p.in = s2.b; p.in_count = e->d_counters + CTR_VIT; p.in_cap = s2.cap;
  p.out = s2.a; p.out_count = e->d_counters + CTR_FWD; p.out_cap = s2.cap;
  if ((rc = fan_out(e))) return rc;
  // widest classes first: their one-warp-per-pair kernels are the long pole of the stage, the narrow ones fill in around them
  if ((rc = launch_fwd(p, nsm * 4, e->cls[N_BLK_CLASSES]))) return rc;
  if (p.use_blk) { for (int c = N_BLK_CLASSES - 1; c >= 0; --c) if ((rc = launch_fwd2(p, c, nsm * 8, e->cls[c]))) return rc; }
  if ((rc = fan_in(e))) return rc;
  CKM_CUDA(cudaEventRecord(e->ev[5], st));
  e->stats.kernel_launches += 3 + (p.use_blk ? 2 * N_BLK_CLASSES : 0);
  s2.fwd_list = s2.a;
  return CKM_OK;
}

}  // namespace ckm

extern "C" {

int ckm_filter_scores(ckm_engine *e, const ckm_models *m, const int32_t *model_idx, int32_t nmodels,
                      const ckm_seqdb *db, float *filtersc_out, float *vit_out, float *fwd_out, uint8_t *passed_out) {
  if (!e || !m || !db || !filtersc_out || !vit_out || !fwd_out || !passed_out) { set_error("ckm_filter_scores: bad argument"); return CKM_EINVAL; }
  cudaSetDevice(e->device);
  if (model_idx == nullptr) nmodels = (int32_t)m->models.size();
  ActiveMasks am; std::vector<int32_t> slot;
  int rc = build_masks(e, m, db, model_idx, nmodels, nullptr, am, slot);
  if (rc) return rc;
  const int64_t n = (int64_t)nmodels * db->nseq;
  float *dfs, *dvit, *dfwd; uint8_t *dpass;
  const size_t nf = (size_t)std::max<int64_t>(n, 1);
  if ((rc = workspace(e, Ws::DenseFiltersc, sizeof(float) * nf, &dfs)) || (rc = workspace(e, Ws::DenseVit, sizeof(float) * nf, &dvit)) ||
      (rc = workspace(e, Ws::DenseFwd, sizeof(float) * nf, &dfwd)) || (rc = workspace(e, Ws::DensePassed, nf + 4, &dpass))) return rc;
  // NaN-fill the float outputs, zero the flags
  CKM_CUDA(cudaMemsetAsync(dfs, 0xff, sizeof(float) * nf, e->stream));
  CKM_CUDA(cudaMemsetAsync(dvit, 0xff, sizeof(float) * nf, e->stream));
  CKM_CUDA(cudaMemsetAsync(dfwd, 0xff, sizeof(float) * nf, e->stream));
  CKM_CUDA(cudaMemsetAsync(dpass, 0, nf + 4, e->stream));
  Stage1 s1; Stage2 s2;
  std::memset(&e->stats, 0, sizeof(e->stats));
  if ((rc = run_stage1(e, m, db, am, n, s1, nullptr))) return rc;
  if ((rc = run_stage2(e, m, db, am, s1, s2, dfs, dvit, dfwd, dpass))) return rc;
  int32_t ctr[CTR_N];
  CKM_CUDA(cudaMemcpyAsync(ctr, e->d_counters, sizeof(ctr), cudaMemcpyDeviceToHost, e->stream));
  CKM_CUDA(cudaMemcpyAsync(filtersc_out, dfs, sizeof(float) * (size_t)n, cudaMemcpyDeviceToHost, e->stream));
  CKM_CUDA(cudaMemcpyAsync(vit_out, dvit, sizeof(float) * (size_t)n, cudaMemcpyDeviceToHost, e->stream));
  CKM_CUDA(cudaMemcpyAsync(fwd_out, dfwd, sizeof(float) * (size_t)n, cudaMemcpyDeviceToHost, e->stream));
  CKM_CUDA(cudaMemcpyAsync(passed_out, dpass, (size_t)n, cudaMemcpyDeviceToHost, e->stream));
  std::vector<Candidate> pass1((size_t)std::min<int64_t>(s1.pass_cap, std::max<int32_t>(1, s1.pass_cap)));
  CKM_CUDA(cudaStreamSynchronize(e->stream));
  if (ctr[CTR_CAND] > s1.cand_cap || ctr[CTR_MSV] > s1.pass_cap) { set_error("candidate queue overflow"); return CKM_ECAPACITY; }
  // MSV pass flags come from the stage-1 pass list
  pass1.resize((size_t)ctr[CTR_MSV]);
  if (!pass1.empty()) CKM_CUDA(cudaMemcpy(pass1.data(), s1.pass, sizeof(Candidate) * pass1.size(), cudaMemcpyDeviceToHost));
  for (const Candidate &c : pass1) passed_out[(int64_t)slot[c.model] * db->nseq + c.seq] |= 1;
  e->stats.n_pairs = n;
  e->stats.n_ssv_cand = (int64_t)ctr[CTR_CAND] + ctr[CTR_SSVRES]; e->stats.n_msv_exact = ctr[CTR_CAND]; e->stats.n_past_msv = ctr[CTR_MSV]; e->stats.n_past_bias = ctr[CTR_BIAS];
  e->stats.n_past_vit = ctr[CTR_VIT]; e->stats.n_past_fwd = ctr[CTR_FWD]; e->stats.n_vit_redo = ctr[CTR_VREDO];
  cudaEventElapsedTime(&e->stats.ms_ssv, e->ev[0], e->ev[1]);
  cudaEventElapsedTime(&e->stats.ms_msv, e->ev[1], e->ev[2]);
  cudaEventElapsedTime(&e->stats.ms_bias, e->ev[2], e->ev[3]);
  cudaEventElapsedTime(&e->stats.ms_vit, e->ev[3], e->ev[4]);
  cudaEventElapsedTime(&e->stats.ms_fwd, e->ev[4], e->ev[5]);
  return CKM_OK;
}

}  // extern "C"

namespace ckm {

constexpr int X_NX_HOST = 6;
struct EnsembleJob;
int ensembles_launch(ckm_engine *e, const ckm_models *m, DomdefParams &p, const std::vector<PairWork> &pairs,
                     const std::vector<Region> &regs, const std::vector<int> &multi_idx, const std::vector<EnsembleCaps> &caps,
                     cudaStream_t st, EnsembleJob **job_out);
int ensembles_collect(EnsembleJob *job, cudaStream_t st, std::vector<std::vector<Envelope>> &out, std::vector<EnsembleCaps> &grow, int *n_over);
void ensembles_abandon(EnsembleJob *job, cudaStream_t st);

static bool use_blocked_kernels() { const char *v = std::getenv("CKM_BLK"); return !(v != nullptr && v[0] == '0'); }
static int vq_of(int M) { return (M <= 64) ? 2 : (M <= 128) ? 4 : (M <= 192) ? 6 : (M <= 256) ? 8 : (M <= 384) ? 12 : (M <= 512) ? 16 : (M <= 640) ? 20 : (M <= 768) ? 24 : (M <= 896) ? 28 : (M <= 1024) ? 32 : 0; }

static int cls_of(int M, bool use_blk) {      // class index: 0..9 lane-block classes, 10 = unblocked kernels
  if (!use_blk) return N_BLK_CLASSES;
  const int q = vq_of(M);
  for (int c = 0; c < N_BLK_CLASSES; ++c) if (BLK_Q[c] == q) return c;
  return N_BLK_CLASSES;
}
// the per-class launches of one stage go to the engine's class streams: fork after the main stream, join back into it
static int fan_out(ckm_engine *e) {
  CKM_CUDA(cudaEventRecord(e->fan_ev, e->stream));
  for (auto &s : e->cls) CKM_CUDA(cudaStreamWaitEvent(s, e->fan_ev, 0));
  return CKM_OK;
}
static int fan_in(ckm_engine *e) {
  for (int c = 0; c < ckm_engine::NCLS; ++c) {
    CKM_CUDA(cudaEventRecord(e->cls_ev[c], e->cls[c]));
    CKM_CUDA(cudaStreamWaitEvent(e->stream, e->cls_ev[c], 0));
  }
  return CKM_OK;
}

static std::vector<float> &logsum_table() {
  static std::vector<float> t = [] {
    std::vector<float> v(16000);
    for (int i = 0; i < 16000; ++i) v[i] = (float)std::log(1.0 + std::exp((double)-i / 1000.0));
    return v;
  }();
  return t;
}


// Envelope rescoring in waves: one matrix (blocked kernels; two for the chunked ones) + specials of scratch per envelope under a fixed budget, every class on its own
// stream.  leave_last: the last wave is left running on the class streams (the caller joins them with fan_in).
struct EnvRunner {
  ckm_engine *e; const ckm_models *m; DomdefParams *p; const std::vector<PairWork> *pairs;
  int64_t budget0;       // floats
  int nsm;
};
static int64_t env_scratch_budget() {
  // fixed scratch budget (the EnvScratch workspace is reused by every later call): 60% of the device shared by the live engines,
  // at most 56 GiB each
  size_t free_b = 0, total_b = 0;
  cudaMemGetInfo(&free_b, &total_b);
  (void)free_b;
  const size_t neng = (size_t)std::max(1, g_live_engines.load());
  return (int64_t)std::min<size_t>(total_b * 6 / 10 / neng, (size_t)56 << 30) / (int64_t)sizeof(float);
}
// floats of scratch one envelope needs (blocked kernels: one matrix, the OA fill overwrites F.B row by row; chunked kernels: two)
static int64_t envelope_need(const ckm_models *m, const PairWork &pw, const Envelope &en, bool use_blk) {
  const int64_t Ld = en.j - en.i + 1, Mpad = ((m->models[pw.model].M + 1) + 31) / 32 * 32 + 32;
  const int64_t vq = use_blk ? vq_of(m->models[pw.model].M) : 0;
  const int64_t width = vq ? 32 * vq : Mpad;
  return (vq ? 1 : 2) * (Ld + 1) * 3 * width + (Ld + 1) * 15 + 64;
}
static int run_envelope_waves(EnvRunner &R, std::vector<Envelope> &ev, Ws envs_key, Ws order_key, bool leave_last) {
  if (ev.empty()) return CKM_OK;
  ckm_engine *e = R.e; const ckm_models *m = R.m; DomdefParams &p = *R.p; const std::vector<PairWork> &pairs = *R.pairs;
  cudaStream_t st = e->stream;
  const int nsm = R.nsm;
  int rc2;
  std::vector<int64_t> need(ev.size());
  std::vector<int8_t> ecls(ev.size());
  for (size_t i = 0; i < ev.size(); ++i) {
    const PairWork &pw = pairs[ev[i].pair];
    need[i] = envelope_need(m, pw, ev[i], p.use_blk != 0);
    ecls[i] = (int8_t)cls_of(m->models[pw.model].M, p.use_blk != 0);
  }
  const int64_t budget = std::max<int64_t>(R.budget0, *std::max_element(need.begin(), need.end()));
  Envelope *d_ev; int32_t *d_ord;
  if ((rc2 = workspace(e, envs_key, sizeof(Envelope) * ev.size(), &d_ev)) || (rc2 = workspace(e, order_key, sizeof(int32_t) * ev.size(), &d_ord))) return rc2;
  p.envs = d_ev; p.env_order = d_ord;
  std::vector<int32_t> eorder(ev.size());
  size_t w0 = 0;
  while (w0 < ev.size()) {
    size_t w1 = w0; int64_t tot = 0;
    while (w1 < ev.size() && (w1 == w0 || tot + need[w1] <= budget)) { ev[w1].scratch_off = tot; tot += need[w1]; ++w1; }
    if ((rc2 = workspace(e, Ws::EnvScratch, sizeof(float) * (size_t)tot, &p.scratch))) return rc2;
    // this wave's envelopes grouped by class, largest first; one stream per class
    for (size_t i = w0; i < w1; ++i) eorder[i] = (int32_t)i;
    std::stable_sort(eorder.begin() + w0, eorder.begin() + w1, [&](int32_t a, int32_t b) { return ecls[a] != ecls[b] ? ecls[a] > ecls[b] : need[a] > need[b]; });
    CKM_CUDA(cudaMemcpyAsync(d_ev + w0, ev.data() + w0, sizeof(Envelope) * (w1 - w0), cudaMemcpyHostToDevice, st));
    CKM_CUDA(cudaMemcpyAsync(d_ord + w0, eorder.data() + w0, sizeof(int32_t) * (w1 - w0), cudaMemcpyHostToDevice, st));
    if ((rc2 = fan_out(e))) return rc2;
    size_t b0 = w0;
    while (b0 < w1) {
      size_t b1 = b0; const int c = ecls[eorder[b0]];
      while (b1 < w1 && ecls[eorder[b1]] == c) ++b1;
      p.env_begin = (int32_t)b0; p.env_end = (int32_t)b1;
      const int cnt = (int)(b1 - b0);
      if (c < N_BLK_CLASSES) rc2 = launch_envelopes2(p, c, std::min<int>(nsm * 8, (cnt + 3) / 4), e->cls[c]);
      else rc2 = launch_envelopes(p, std::min<int>(nsm * 4, (cnt + FWD_WARPS - 1) / FWD_WARPS), e->cls[c]);
      if (rc2) return rc2;
      e->stats.kernel_launches++;
      b0 = b1;
    }
    CKM_CUDA(cudaStreamSynchronize(st));          // the two copies above have read the host vectors
    if (w1 < ev.size() || !leave_last) {
      if ((rc2 = fan_in(e))) return rc2;
      CKM_CUDA(cudaStreamSynchronize(st));
    }
    w0 = w1;
  }
  return CKM_OK;
}

struct HostHit { int pair; HitOut h; int first_dom, ndom_slots; };

// CKM_TRACE=1: host-side wall-clock marks of one search on stderr (where the time between the CUDA events goes)
struct Trace {
  bool on; std::chrono::steady_clock::time_point t0, last;
  Trace() { const char *v = std::getenv("CKM_TRACE"); on = (v != nullptr && v[0] == '1'); t0 = last = std::chrono::steady_clock::now(); }
  void mark(const char *what) {
    if (!on) return;
    const auto now = std::chrono::steady_clock::now();
    std::fprintf(stderr, "[ckm trace] %-28s +%8.3f ms  (%9.3f)\n", what, std::chrono::duration<double, std::milli>(now - last).count(),
                 std::chrono::duration<double, std::milli>(now - t0).count());
    last = now;
  }
};

static int do_search(ckm_engine *e, const ckm_models *m, const int32_t *model_idx, int32_t nmodels, const int64_t *bin_model_offsets,
                     const ckm_seqdb *db, double Ecut, double domEcut, ckm_hit **hits_out, int64_t *nhits_out) {
  if (!e || !m || !db || !hits_out || !nhits_out) { set_error("ckm_search: bad argument"); return CKM_EINVAL; }
  cudaSetDevice(e->device);
  cudaStream_t st = e->stream;
  *hits_out = nullptr; *nhits_out = 0;
  const int ndb = (int)m->models.size();
  if (model_idx == nullptr && bin_model_offsets == nullptr) nmodels = ndb;
  ActiveMasks am; std::vector<int32_t> slot;
  int rc = build_masks(e, m, db, model_idx, nmodels, bin_model_offsets, am, slot);
  if (rc) return rc;
  // query order per bin (for output ordering) and the number of pairs
  int64_t n_pairs = 0;
  std::vector<std::vector<int32_t>> qorder(bin_model_offsets ? db->nbins : 1);
  if (bin_model_offsets) {
    for (int b = 0; b < db->nbins; ++b) {
      qorder[b].assign(ndb, -1);
      for (int64_t i = bin_model_offsets[b]; i < bin_model_offsets[b + 1]; ++i) qorder[b][model_idx[i]] = (int32_t)(i - bin_model_offsets[b]);
      n_pairs += (int64_t)db->bin_nseq[b] * (bin_model_offsets[b + 1] - bin_model_offsets[b]);
    }
  } else {
    qorder[0] = slot;
    n_pairs = (int64_t)db->nseq * nmodels;
  }
  std::memset(&e->stats, 0, sizeof(e->stats));
  if (n_pairs > ((int64_t)1 << 40)) { set_error("ckm_search: more than 2^40 (ORF x HMM) pairs in one call; search fewer bins per call"); return CKM_ECAPACITY; }
  CKM_CUDA(cudaEventRecord(e->ev[8], st));
  Trace tr;
  Stage1 s1; Stage2 s2;
  int32_t ctr[CTR_N];
  unsigned long long cells = 0;
  for (int attempt = 0;; ++attempt) {
    // a candidate-dense input (many pairs past SSV) overflows the default queues: the cascade is re-run with larger ones
    if ((rc = run_stage1(e, m, db, am, std::max<int64_t>(n_pairs, 1), s1, nullptr, attempt))) return rc;
    if ((rc = run_stage2(e, m, db, am, s1, s2, nullptr, nullptr, nullptr, nullptr))) return rc;
    CKM_CUDA(cudaMemcpyAsync(ctr, e->d_counters, sizeof(ctr), cudaMemcpyDeviceToHost, st));
    CKM_CUDA(cudaMemcpyAsync(&cells, s1.cells, sizeof(cells), cudaMemcpyDeviceToHost, st));
    CKM_CUDA(cudaStreamSynchronize(st));
    const bool over = ctr[CTR_CAND] > s1.cand_cap || ctr[CTR_MSV] > s1.pass_cap || ctr[CTR_BIAS] > s2.cap || ctr[CTR_VIT] > s2.cap || ctr[CTR_FWD] > s2.cap ||
                      ctr[CTR_VREDO] > s2.cap;
    if (!over) break;
    if (attempt >= 2 || (s1.cand_cap >= std::min<int64_t>(n_pairs, QUEUE_MAX) && s1.pass_cap >= std::min<int64_t>(n_pairs, QUEUE_MAX))) {
      set_error("candidate queue overflow in the filter cascade: more than 2^30 candidate pairs in one batch; search fewer bins per call");
      return CKM_ECAPACITY;
    }
    e->stats.n_queue_retries++;
  }
  tr.mark("filters done");
  e->stats.n_pairs = n_pairs; e->stats.n_cells = (int64_t)cells;
  e->stats.n_ssv_cand = (int64_t)ctr[CTR_CAND] + ctr[CTR_SSVRES]; e->stats.n_msv_exact = ctr[CTR_CAND]; e->stats.n_past_msv = ctr[CTR_MSV]; e->stats.n_past_bias = ctr[CTR_BIAS];
  e->stats.n_past_vit = ctr[CTR_VIT]; e->stats.n_past_fwd = ctr[CTR_FWD]; e->stats.n_vit_redo = ctr[CTR_VREDO];
  const int npairs = ctr[CTR_FWD];
  std::vector<Candidate> fl((size_t)npairs);
  if (npairs) CKM_CUDA(cudaMemcpy(fl.data(), s2.fwd_list, sizeof(Candidate) * fl.size(), cudaMemcpyDeviceToHost));
  std::sort(fl.begin(), fl.end(), [](const Candidate &a, const Candidate &b) { return a.seq != b.seq ? a.seq < b.seq : a.model < b.model; });

  std::vector<PairWork> pairs((size_t)npairs);
  int64_t rows = 0;
  for (int i = 0; i < npairs; ++i) {
    PairWork &pw = pairs[i];
    pw.seq = fl[i].seq; pw.model = fl[i].model; pw.L = db->len[pw.seq];
    pw.first_dom = 0; pw.ndom_slots = 0; pw.fwdsc = fl[i].fwdsc; pw.filtersc = fl[i].filtersc; pw.usc = fl[i].usc;
    pw.row_off = rows; rows += pw.L + 1;
  }
  const int nsm = e->prop.multiProcessorCount;
  std::vector<DomainOut> doms; std::vector<HitOut> hout((size_t)npairs);
  CKM_CUDA(cudaEventRecord(e->ev[6], st));
  tr.mark("pair list sorted");
  if (npairs > 0) {
    const size_t rws = (size_t)std::max<int64_t>(rows, 1);
    DomdefParams p{};
    PairWork *dpairs; float *dtbl;
    const int region_cap = npairs * 8 + 1024;
    if ((rc = workspace(e, Ws::Pairs, sizeof(PairWork) * pairs.size(), &dpairs)) || (rc = workspace(e, Ws::Xf, sizeof(float) * rws * X_NX_HOST, &p.xf)) ||
        (rc = workspace(e, Ws::Xb, sizeof(float) * rws * X_NX_HOST, &p.xb)) || (rc = workspace(e, Ws::Vec, sizeof(float) * rws * 4, &p.btot)) ||
        (rc = workspace(e, Ws::LogsumTbl, sizeof(float) * 16000, &dtbl)) || (rc = workspace(e, Ws::Regions, sizeof(Region) * (size_t)region_cap, &p.regions))) return rc;
    CKM_CUDA(cudaMemcpyAsync(dpairs, pairs.data(), sizeof(PairWork) * pairs.size(), cudaMemcpyHostToDevice, st));
    CKM_CUDA(cudaMemcpyAsync(dtbl, logsum_table().data(), sizeof(float) * 16000, cudaMemcpyHostToDevice, st));
    CKM_CUDA(cudaMemsetAsync(e->d_counters + CTR_ENV, 0, sizeof(int32_t), st));
    p.res = db->d_res; p.off = db->d_off; p.nullsc = db->d_nullsc; p.ms = m->d_scalars; p.rfv = m->d_rfv; p.tfv = m->d_tfv;
    p.pairs = dpairs; p.npairs = npairs;
    p.etot = p.btot + rws; p.mocc = p.etot + rws; p.n2sc = p.mocc + rws;
    p.region_count = e->d_counters + CTR_ENV; p.region_cap = region_cap;
    p.logsum_tbl = dtbl;
    p.row_elems = ((m->maxM + 31) / 32) * 32 + 64;
    p.tfb = m->d_tfb; p.rfb = m->d_rfb; p.use_blk = use_blocked_kernels() ? 1 : 0;
    {
      // pairs grouped by class (widest class first: it is the long pole), longest target first inside a class; every class runs on its own stream
      std::vector<int32_t> order((size_t)npairs);
      std::vector<int8_t> pcls((size_t)npairs);
      for (int i = 0; i < npairs; ++i) { order[i] = i; pcls[i] = (int8_t)cls_of(m->models[pairs[i].model].M, p.use_blk != 0); }
      std::stable_sort(order.begin(), order.end(), [&](int32_t a, int32_t b) { return pcls[a] != pcls[b] ? pcls[a] > pcls[b] : pairs[a].L > pairs[b].L; });
      int32_t *dporder;
      if ((rc = workspace(e, Ws::PairOrder, sizeof(int32_t) * order.size(), &dporder))) return rc;
      CKM_CUDA(cudaMemcpyAsync(dporder, order.data(), sizeof(int32_t) * order.size(), cudaMemcpyHostToDevice, st));
      p.pair_order = dporder;
      if ((rc = fan_out(e))) return rc;
      int b0 = 0;
      while (b0 < npairs) {
        int b1 = b0; const int c = pcls[order[b0]];
        while (b1 < npairs && pcls[order[b1]] == c) ++b1;
        p.pair_begin = b0; p.pair_end = b1;
        const int cnt = b1 - b0;
        if (c < N_BLK_CLASSES) rc = launch_regions2(p, c, std::min(nsm * 8, (cnt + 3) / 4), e->cls[c]);
        else rc = launch_regions(p, std::min(nsm * 4, (cnt + FWD_WARPS - 1) / FWD_WARPS), e->cls[c]);
        if (rc) return rc;
        e->stats.kernel_launches++;
        b0 = b1;
      }
      if ((rc = fan_in(e))) return rc;
      CKM_CUDA(cudaStreamSynchronize(st));   // `order` is read by the copy above
      tr.mark("regions kernels");
    }
    int32_t nreg = 0;
    CKM_CUDA(cudaMemcpyAsync(&nreg, e->d_counters + CTR_ENV, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    CKM_CUDA(cudaStreamSynchronize(st));
    if (nreg > region_cap) { set_error("region queue overflow"); return CKM_ECAPACITY; }
    std::vector<Region> regs((size_t)nreg);
    if (nreg) CKM_CUDA(cudaMemcpy(regs.data(), p.regions, sizeof(Region) * regs.size(), cudaMemcpyDeviceToHost));
    std::sort(regs.begin(), regs.end(), [](const Region &a, const Region &b) { return a.pair != b.pair ? a.pair < b.pair : a.i < b.i; });
    tr.mark("regions sorted");
    // Domain slots.  Regions are sorted by (pair, start), so a pair's slots are contiguous and in sequence order: one slot
    // per single-domain region, ENS_MAXENV per multi-domain region (the ensemble decides how many it fills; unused slots
    // keep ok = 0 and are skipped by every consumer).  Fixing the slots before the ensemble has run lets the envelopes of
    // the single-domain regions be rescored WHILE the trace ensemble of the multi-domain ones is still sampling.
    // A region that turns out to hold more domains than its slots (or more sampled segments than its clustering buffers)
    // reports what it needs, and the phase is repeated from here with that region's capacities raised.
    std::vector<int> multi_idx;
    for (int r = 0; r < nreg; ++r) if (regs[r].multi) multi_idx.push_back(r);
    std::vector<EnsembleCaps> caps(multi_idx.size(), ENS_DEFAULT_CAPS);
    std::vector<int32_t> reg_slot((size_t)nreg);
    for (int pass = 0;; ++pass) {
    int32_t nslots = 0;
    for (auto &pw : pairs) { pw.ndom_slots = 0; pw.first_dom = 0; }
    for (int r = 0, mi = 0; r < nreg; ++r) {
      PairWork &pw = pairs[regs[r].pair];
      if (pw.ndom_slots == 0) pw.first_dom = nslots;
      reg_slot[r] = nslots;
      const int k = regs[r].multi ? caps[mi++].envelopes : 1;
      nslots += k; pw.ndom_slots += k;
    }
    doms.assign((size_t)nslots, DomainOut{});
    std::vector<Envelope> envs1, envs2;
    for (int r = 0; r < nreg; ++r)
      if (!regs[r].multi) { Envelope en{}; en.pair = regs[r].pair; en.i = regs[r].i; en.j = regs[r].j; en.slot = reg_slot[r]; envs1.push_back(en); }
    if (nslots > 0) {
      DomainOut *ddoms; HitOut *dhits;
      if ((rc = workspace(e, Ws::Doms, sizeof(DomainOut) * (size_t)nslots, &ddoms)) || (rc = workspace(e, Ws::Hits, sizeof(HitOut) * pairs.size(), &dhits))) return rc;
      CKM_CUDA(cudaMemsetAsync(ddoms, 0, sizeof(DomainOut) * (size_t)nslots, st));
      CKM_CUDA(cudaMemcpyAsync(dpairs, pairs.data(), sizeof(PairWork) * pairs.size(), cudaMemcpyHostToDevice, st));
      p.doms = ddoms;
      EnvRunner R{e, m, &p, &pairs, env_scratch_budget(), nsm};
      // The trace ensemble of the multi-domain regions (one warp per region, latency-bound, its own stream) runs next to the
      // envelope kernels of the single-domain regions (class streams).  Next to them its dependent loads take 2-3x longer than
      // alone.  When the envelopes need more than one wave of scratch (large batches) it is queued FIRST and has all the waves to
      // hide under (32-bin batch: domain stage 501 -> 485 ms); with a single wave it is queued after the envelope kernels and takes
      // the SMs as they drain.  CKM_ENS_FIRST=1 / 0 forces one order.
      EnsembleJob *job = nullptr;
      static const int ens_knob = [] { const char *v = std::getenv("CKM_ENS_FIRST"); return v == nullptr ? -1 : (v[0] == '0' ? 0 : 1); }();
      bool ens_first = (ens_knob == 1);
      if (ens_knob < 0 && !multi_idx.empty()) {
        int64_t tot = 0;
        for (const Envelope &en : envs1) tot += envelope_need(m, pairs[en.pair], en, p.use_blk != 0);
        ens_first = tot > R.budget0;
      }
      if (ens_first && !multi_idx.empty()) {
        CKM_CUDA(cudaEventRecord(e->fan_ev, st));
        CKM_CUDA(cudaStreamWaitEvent(e->aux, e->fan_ev, 0));
        if ((rc = ensembles_launch(e, m, p, pairs, regs, multi_idx, caps, e->aux, &job))) { ensembles_abandon(job, e->aux); return rc; }
      }
      if ((rc = run_envelope_waves(R, envs1, Ws::Envs1, Ws::EnvOrder1, !multi_idx.empty()))) { if (job) ensembles_abandon(job, e->aux); return rc; }
      tr.mark("envelope batch 1 launched");
      if (!multi_idx.empty()) {
        if (!ens_first) {
          CKM_CUDA(cudaEventRecord(e->fan_ev, st));
          CKM_CUDA(cudaStreamWaitEvent(e->aux, e->fan_ev, 0));
          if ((rc = ensembles_launch(e, m, p, pairs, regs, multi_idx, caps, e->aux, &job))) { ensembles_abandon(job, e->aux); return rc; }
        }
        if (!envs1.empty()) { if ((rc = fan_in(e))) { ensembles_abandon(job, e->aux); return rc; } CKM_CUDA(cudaStreamSynchronize(st)); }
      }
      if (job != nullptr) {
        std::vector<std::vector<Envelope>> multi_envs;
        std::vector<EnsembleCaps> grow;
        int n_over = 0;
        if ((rc = ensembles_collect(job, e->aux, multi_envs, grow, &n_over))) return rc;
        tr.mark("batch 1 + ensemble done");
        if (n_over > 0) {
          if (pass >= 3) { set_error("a multi-domain region keeps outgrowing the capacities it asked for"); return CKM_ECAPACITY; }
          for (size_t mi = 0; mi < caps.size(); ++mi) if (grow[mi].segments) caps[mi] = grow[mi];
          e->stats.n_queue_retries++;
          continue;
        }
        for (size_t mi = 0; mi < multi_idx.size(); ++mi) {
          int c = 0;
          for (Envelope en : multi_envs[mi]) { en.slot = reg_slot[multi_idx[mi]] + c++; envs2.push_back(en); }     // no more than the region's slots (ensembles_collect)
        }
        if ((rc = run_envelope_waves(R, envs2, Ws::Envs2, Ws::EnvOrder2, false))) return rc;
        tr.mark("envelope batch 2 done");
      }
      p.hits = dhits;
      if ((rc = launch_scores(p, (npairs + 127) / 128, st))) return rc;
      e->stats.kernel_launches++;
      CKM_CUDA(cudaMemcpyAsync(doms.data(), ddoms, sizeof(DomainOut) * doms.size(), cudaMemcpyDeviceToHost, st));
      CKM_CUDA(cudaMemcpyAsync(hout.data(), dhits, sizeof(HitOut) * hout.size(), cudaMemcpyDeviceToHost, st));
      CKM_CUDA(cudaStreamSynchronize(st));
    } else {
      for (auto &h : hout) std::memset(&h, 0, sizeof(h));
    }
    break;
    }   // pass
  }
  CKM_CUDA(cudaEventRecord(e->ev[7], st));
  CKM_CUDA(cudaEventSynchronize(e->ev[7]));
  tr.mark("scores + downloads");

  // ---- thresholds, ordering, rows (bookkeeping on the hit list; hmmsearch's output phase) ----
  struct Key { int bin, q, pair; double lnP; int seq; };
  std::vector<Key> keys;
  for (int i = 0; i < npairs; ++i) {
    if (!hout[i].valid) continue;
    const int b = db->bin_of_seq[pairs[i].seq];
    const int q = (bin_model_offsets ? qorder[b] : qorder[0])[pairs[i].model];
    keys.push_back(Key{b, q, i, hout[i].lnP, pairs[i].seq});
  }
  std::sort(keys.begin(), keys.end(), [](const Key &a, const Key &b) {
    if (a.bin != b.bin) return a.bin < b.bin;
    if (a.q != b.q) return a.q < b.q;
    if (a.lnP != b.lnP) return a.lnP < b.lnP;
    return a.seq < b.seq;
  });
  std::vector<ckm_hit> rows_out;
  size_t g0 = 0;
  int64_t n_dom = 0;
  for (size_t i = 0; i < doms.size(); ++i) if (doms[i].ok) n_dom++;
  while (g0 < keys.size()) {
    size_t g1 = g0;
    while (g1 < keys.size() && keys[g1].bin == keys[g0].bin && keys[g1].q == keys[g0].q) ++g1;
    const double Z = (double)db->bin_nseq[keys[g0].bin];
    double domZ = 0.0;
    for (size_t k = g0; k < g1; ++k) if (std::exp(keys[k].lnP) * Z <= Ecut) domZ += 1.0;
    for (size_t k = g0; k < g1; ++k) {
      if (!(std::exp(keys[k].lnP) * Z <= Ecut)) continue;
      const PairWork &pw = pairs[keys[k].pair];
      const HitOut &h = hout[keys[k].pair];
      int nrep = 0;
      for (int d = pw.first_dom; d < pw.first_dom + pw.ndom_slots; ++d)
        if (doms[d].ok && std::exp(doms[d].lnP) * domZ <= domEcut) nrep++;
      int nd = 0;
      for (int d = pw.first_dom; d < pw.first_dom + pw.ndom_slots; ++d) {
        const DomainOut &dm = doms[d];
        if (!dm.ok || !(std::exp(dm.lnP) * domZ <= domEcut)) continue;
        ckm_hit r;
        std::memset(&r, 0, sizeof(r));
        r.bin = keys[k].bin; r.seq = pw.seq; r.model = pw.model; r.tlen = pw.L; r.qlen = m->models[pw.model].M;
        r.dom = ++nd; r.ndom = nrep;
        r.hmm_from = dm.hmmfrom; r.hmm_to = dm.hmmto; r.ali_from = dm.sqfrom; r.ali_to = dm.sqto; r.env_from = dm.ienv; r.env_to = dm.jenv;
        r.full_score = h.score; r.full_bias = h.pre_score - h.score;
        r.dom_score = dm.bitscore; r.dom_bias = (float)((double)dm.dombias * 1.44269504088896341);
        r.acc = (float)(dm.oasc / (1.0 + std::fabs((float)(dm.jenv - dm.ienv))));
        r.full_evalue = std::exp(h.lnP) * Z; r.c_evalue = std::exp(dm.lnP) * domZ; r.i_evalue = std::exp(dm.lnP) * Z;
        r.full_lnP = h.lnP; r.dom_lnP = dm.lnP;
        rows_out.push_back(r);
      }
    }
    g0 = g1;
  }
  tr.mark("rows assembled");
  e->stats.n_hits_seq = (int64_t)keys.size(); e->stats.n_domains = n_dom; e->stats.n_reported = (int64_t)rows_out.size();
  cudaEventElapsedTime(&e->stats.ms_ssv, e->ev[0], e->ev[1]);
  cudaEventElapsedTime(&e->stats.ms_msv, e->ev[1], e->ev[2]);
  cudaEventElapsedTime(&e->stats.ms_bias, e->ev[2], e->ev[3]);
  cudaEventElapsedTime(&e->stats.ms_vit, e->ev[3], e->ev[4]);
  cudaEventElapsedTime(&e->stats.ms_fwd, e->ev[4], e->ev[5]);
  cudaEventElapsedTime(&e->stats.ms_domdef, e->ev[6], e->ev[7]);
  cudaEventElapsedTime(&e->stats.ms_total, e->ev[8], e->ev[7]);
  if (!rows_out.empty()) {
    ckm_hit *out = (ckm_hit *)std::malloc(sizeof(ckm_hit) * rows_out.size());
    if (!out) { set_error("out of host memory"); return CKM_ENOMEM; }
    std::memcpy(out, rows_out.data(), sizeof(ckm_hit) * rows_out.size());
    *hits_out = out;
  }
  *nhits_out = (int64_t)rows_out.size();
  return CKM_OK;
}

}  // namespace ckm

extern "C" {

int ckm_search(ckm_engine *e, const ckm_models *m, const int32_t *model_idx, int32_t nmodels,
               const ckm_seqdb *db, double E, double domE, ckm_hit **hits_out, int64_t *nhits_out) {
  return do_search(e, m, model_idx, nmodels, nullptr, db, E, domE, hits_out, nhits_out);
}

int ckm_search_per_bin(ckm_engine *e, const ckm_models *m, const int32_t *model_idx, const int64_t *bin_model_offsets,
                       const ckm_seqdb *db, double E, double domE, ckm_hit **hits_out, int64_t *nhits_out) {
  if (!model_idx || !bin_model_offsets) { set_error("ckm_search_per_bin: bad argument"); return CKM_EINVAL; }
  return do_search(e, m, model_idx, 0, bin_model_offsets, db, E, domE, hits_out, nhits_out);
}

// domtblout writer: the 22 columns + description CheckM's HMMERParser.readHitsDOM splits (checkm/hmmer.py:184-200)
int ckm_write_domtblout(const ckm_models *m, const ckm_hit *hits, int64_t nhits, int32_t bin, int32_t seq_base,
                        const char *const *names, const char *const *descs, const char *path) {
  if (!m || (!hits && nhits > 0) || !names || !path) { set_error("ckm_write_domtblout: bad argument"); return CKM_EINVAL; }
  FILE *fp = std::fopen(path, "w");
  if (!fp) { set_error(std::string("cannot write ") + path); return CKM_EIO; }
  int tnamew = 20, qnamew = 20, qaccw = 10, taccw = 10;
  for (int64_t i = 0; i < nhits; ++i) {
    if (hits[i].bin != bin) continue;
    const Model &md = m->models[hits[i].model];
    tnamew = std::max<int>(tnamew, (int)std::strlen(names[hits[i].seq - seq_base]));
    qnamew = std::max<int>(qnamew, (int)md.name.size());
    qaccw = std::max<int>(qaccw, (int)md.acc.size());
  }
  std::fprintf(fp, "#%*s %22s %40s %11s %11s %11s\n", tnamew + qnamew - 1 + 15 + taccw + qaccw, "", "--- full sequence ---",
               "-------------- this domain -------------", "hmm coord", "ali coord", "env coord");
  std::fprintf(fp, "#%-*s %-*s %5s %-*s %-*s %5s %9s %6s %5s %3s %3s %9s %9s %6s %5s %5s %5s %5s %5s %5s %5s %4s %s\n",
               tnamew - 1, " target name", taccw, "accession", "tlen", qnamew, "query name", qaccw, "accession", "qlen",
               "E-value", "score", "bias", "#", "of", "c-Evalue", "i-Evalue", "score", "bias", "from", "to", "from", "to", "from", "to", "acc", "description of target");
  std::fprintf(fp, "#%*s %*s ----- %*s %*s ----- --------- ------ ----- --- --- --------- --------- ------ ----- ----- ----- ----- ----- ----- ----- ---- ---------------------\n",
               tnamew - 1, "-------------------", taccw, "----------", qnamew, "--------------------", qaccw, "----------");
  for (int64_t i = 0; i < nhits; ++i) {
    const ckm_hit &h = hits[i];
    if (h.bin != bin) continue;
    const Model &md = m->models[h.model];
    const char *desc = (descs && descs[h.seq - seq_base] && descs[h.seq - seq_base][0]) ? descs[h.seq - seq_base] : "-";
    std::fprintf(fp, "%-*s %-*s %5d %-*s %-*s %5d %9.2g %6.1f %5.1f %3d %3d %9.2g %9.2g %6.1f %5.1f %5d %5d %5d %5d %5d %5d %4.2f %s\n",
                 tnamew, names[h.seq - seq_base], taccw, "-", h.tlen, qnamew, md.name.c_str(), qaccw, md.acc.empty() ? "-" : md.acc.c_str(), h.qlen,
                 h.full_evalue, h.full_score, h.full_bias, h.dom, h.ndom, h.c_evalue, h.i_evalue, h.dom_score, h.dom_bias,
                 h.hmm_from, h.hmm_to, h.ali_from, h.ali_to, h.env_from, h.env_to, h.acc, desc);
  }
  std::fprintf(fp, "#\n# Program:         checkm_b200 (libckm.so)\n# Pipeline mode:   SEARCH\n# [ok]\n");
  std::fclose(fp);
  return CKM_OK;
}

int ckm_viterbi_scores(ckm_engine *e, const ckm_models *m, const int32_t *model_idx, int32_t nmodels,
                       const ckm_seqdb *db, int32_t mode, float *vit_out) {
  if (!e || !m || !db || !vit_out) { set_error("ckm_viterbi_scores: bad argument"); return CKM_EINVAL; }
  cudaSetDevice(e->device);
  cudaStream_t st = e->stream;
  const int ndb = (int)m->models.size();
  if (model_idx == nullptr) nmodels = ndb;
  const int64_t n = (int64_t)nmodels * db->nseq;
  if (n > ((int64_t)1 << 30)) { set_error("ckm_viterbi_scores: too many pairs for one call"); return CKM_ECAPACITY; }
  ActiveMasks am; std::vector<int32_t> slot;
  int rc = build_masks(e, m, db, model_idx, nmodels, nullptr, am, slot);
  if (rc) return rc;
  std::vector<int32_t> slot_model((size_t)std::max(nmodels, 1));
  for (int i = 0; i < nmodels; ++i) slot_model[i] = model_idx ? model_idx[i] : i;
  const size_t nf = (size_t)std::max<int64_t>(n, 1);
  int32_t *dsm; Candidate *din, *dout, *dredo; float *dvit;
  if ((rc = workspace(e, Ws::SlotModel, sizeof(int32_t) * slot_model.size(), &dsm)) || (rc = workspace(e, Ws::ListA, sizeof(Candidate) * nf, &din)) ||
      (rc = workspace(e, Ws::ListB, sizeof(Candidate) * nf, &dout)) || (rc = workspace(e, Ws::Redo, sizeof(Candidate) * nf, &dredo)) ||
      (rc = workspace(e, Ws::DenseVit, sizeof(float) * nf, &dvit))) return rc;
  CKM_CUDA(cudaMemcpyAsync(dsm, slot_model.data(), sizeof(int32_t) * slot_model.size(), cudaMemcpyHostToDevice, st));
  CKM_CUDA(cudaMemsetAsync(e->d_counters, 0, CTR_N * sizeof(int32_t), st));
  CKM_CUDA(cudaMemsetAsync(dvit, 0xff, sizeof(float) * nf, st));
  std::memset(&e->stats, 0, sizeof(e->stats));
  if (n > 0) {
    if ((rc = launch_all_pairs(din, e->d_counters + CTR_BIAS, dsm, nmodels, db->nseq, st))) return rc;
    const int nsm = e->prop.multiProcessorCount;
    FilterParams p{};
    p.res = db->d_res; p.off = db->d_off; p.len = db->d_len; p.lenA = db->d_lenA; p.lenB = db->d_lenB; p.tmove_w = db->d_tmove_w;
    p.ms = m->d_scalars; p.bias_eo = m->d_bias_eo; p.rwv = m->d_rwv; p.twv = m->d_twv; p.rfv = m->d_rfv; p.tfv = m->d_tfv;
    p.twb = m->d_twb; p.rwb = m->d_rwb; p.tfb = m->d_tfb; p.rfb = m->d_rfb; p.twp = m->d_twp; p.rwp = m->d_rwp;
    p.row_elems = ((m->maxM + 31) / 32) * 32 + 64;
    p.F1 = 0.02; p.F2 = 1e-3; p.F3 = 1e-5; p.use_blk = (mode == 2) ? 0 : 1;      // mode 2: every pair through the chunked shared-memory kernel
    p.dense_vit = dvit; p.model_slot = am.model_slot; p.nseq = db->nseq;
    p.redo = dredo; p.redo_count = e->d_counters + CTR_VREDO; p.redo_cap = (int32_t)nf;
    p.in = din; p.in_count = e->d_counters + CTR_BIAS; p.in_cap = (int32_t)nf;
    p.out = dout; p.out_count = e->d_counters + CTR_VIT; p.out_cap = (int32_t)nf;
    if (mode == 0) {
      p.vit_work = e->d_counters + CTR_VWORK;
      if ((rc = fan_out(e))) return rc;
      for (int c = 0; c < N_BLK_CLASSES; ++c) if ((rc = launch_vitp(p, c, nsm * 8, e->cls[c]))) return rc;
      if ((rc = fan_in(e))) return rc;
      p.in = dredo; p.in_count = e->d_counters + CTR_VREDO;
    }
    if ((rc = fan_out(e))) return rc;
    if (p.use_blk) { for (int c = 0; c < N_BLK_CLASSES; ++c) if ((rc = launch_vit2(p, c, nsm * 8, e->cls[c]))) return rc; }
    if ((rc = launch_vit(p, nsm * 4, e->cls[N_BLK_CLASSES]))) return rc;
    if ((rc = fan_in(e))) return rc;
  }
  int32_t ctr[CTR_N];
  CKM_CUDA(cudaMemcpyAsync(ctr, e->d_counters, sizeof(ctr), cudaMemcpyDeviceToHost, st));
  CKM_CUDA(cudaMemcpyAsync(vit_out, dvit, sizeof(float) * (size_t)n, cudaMemcpyDeviceToHost, st));
  CKM_CUDA(cudaStreamSynchronize(st));
  e->stats.n_pairs = n; e->stats.n_past_bias = ctr[CTR_BIAS]; e->stats.n_past_vit = ctr[CTR_VIT]; e->stats.n_vit_redo = ctr[CTR_VREDO];
  return CKM_OK;
}

int ckm_msv_scores(ckm_engine *e, const ckm_models *m, const int32_t *model_idx, int32_t nmodels,
                   const ckm_seqdb *db, int32_t *xj_out) {
  if (!e || !m || !db || !xj_out) { set_error("ckm_msv_scores: bad argument"); return CKM_EINVAL; }
  cudaSetDevice(e->device);
  if (model_idx == nullptr) nmodels = (int32_t)m->models.size();
  ActiveMasks am; std::vector<int32_t> slot;
  int rc = build_masks(e, m, db, model_idx, nmodels, nullptr, am, slot);
  if (rc) return rc;
  const int64_t n = (int64_t)nmodels * db->nseq;
  int32_t *dense;
  if ((rc = workspace(e, Ws::DenseXj, sizeof(int32_t) * (size_t)std::max<int64_t>(n, 1), &dense))) return rc;
  CKM_CUDA(cudaMemsetAsync(dense, 0xff, sizeof(int32_t) * (size_t)n, e->stream));
  Stage1 s1;
  std::memset(&e->stats, 0, sizeof(e->stats));
  if ((rc = run_stage1(e, m, db, am, n, s1, dense))) return rc;
  int32_t ctr[CTR_N];
  CKM_CUDA(cudaMemcpyAsync(ctr, e->d_counters, sizeof(ctr), cudaMemcpyDeviceToHost, e->stream));
  unsigned long long cells = 0;
  CKM_CUDA(cudaMemcpyAsync(&cells, s1.cells, sizeof(cells), cudaMemcpyDeviceToHost, e->stream));
  CKM_CUDA(cudaMemcpyAsync(xj_out, dense, sizeof(int32_t) * (size_t)n, cudaMemcpyDeviceToHost, e->stream));
  CKM_CUDA(cudaStreamSynchronize(e->stream));
  if (ctr[CTR_CAND] > s1.cand_cap || ctr[CTR_MSV] > s1.pass_cap) { set_error("candidate queue overflow"); return CKM_ECAPACITY; }
  e->stats.n_pairs = n; e->stats.n_cells = (int64_t)cells;
  e->stats.n_ssv_cand = (int64_t)ctr[CTR_CAND] + ctr[CTR_SSVRES]; e->stats.n_msv_exact = ctr[CTR_CAND]; e->stats.n_past_msv = ctr[CTR_MSV];
  cudaEventElapsedTime(&e->stats.ms_ssv, e->ev[0], e->ev[1]);
  cudaEventElapsedTime(&e->stats.ms_msv, e->ev[1], e->ev[2]);
  return CKM_OK;
}

}  // extern "C"

namespace ckm {

// hmmalign: every sequence against one model, as one full-length envelope in unihit local mode (what `hmmalign` configures:
// Forward, Backward, posterior decoding, optimal-accuracy fill and traceback); the traceback's state per residue is the output.
// A sequence that carries a second strong copy of the domain cannot be scored as ONE unihit envelope in scaled fp32 (the
// Backward pass overflows where the Forward pass has underflowed); such a sequence is aligned over the envelope of its
// best-scoring domain as the search pipeline defines it, the rest of it being flank.
static int align_pass(ckm_engine *e, const ckm_models *m, const ckm_seqdb *db, std::vector<PairWork> &pairs, std::vector<Envelope> &envs,
                      int64_t rows, std::vector<int32_t> &trace, std::vector<DomainOut> &doms) {
  cudaStream_t st = e->stream;
  const int nsm = e->prop.multiProcessorCount;
  DomdefParams p{};
  PairWork *dpairs;
  int rc;
  const size_t rws = (size_t)rows;
  if ((rc = workspace(e, Ws::Pairs, sizeof(PairWork) * pairs.size(), &dpairs)) || (rc = workspace(e, Ws::Vec, sizeof(float) * rws, &p.n2sc)) ||
      (rc = workspace(e, Ws::AlignTrace, sizeof(int32_t) * rws, &p.trace)) || (rc = workspace(e, Ws::Doms, sizeof(DomainOut) * pairs.size(), &p.doms))) return rc;
  CKM_CUDA(cudaMemcpyAsync(dpairs, pairs.data(), sizeof(PairWork) * pairs.size(), cudaMemcpyHostToDevice, st));
  CKM_CUDA(cudaMemsetAsync(p.n2sc, 0, sizeof(float) * rws, st));
  CKM_CUDA(cudaMemsetAsync(p.trace, 0, sizeof(int32_t) * rws, st));
  CKM_CUDA(cudaMemsetAsync(p.doms, 0, sizeof(DomainOut) * pairs.size(), st));
  p.res = db->d_res; p.off = db->d_off; p.nullsc = db->d_nullsc; p.ms = m->d_scalars; p.rfv = m->d_rfv; p.tfv = m->d_tfv;
  p.pairs = dpairs; p.npairs = (int32_t)pairs.size();
  p.row_elems = ((m->maxM + 31) / 32) * 32 + 64;
  p.tfb = m->d_tfb; p.rfb = m->d_rfb; p.use_blk = use_blocked_kernels() ? 1 : 0;
  EnvRunner R{e, m, &p, &pairs, env_scratch_budget(), nsm};
  if ((rc = run_envelope_waves(R, envs, Ws::Envs1, Ws::EnvOrder1, false))) return rc;
  trace.resize(rws);
  doms.resize(pairs.size());
  CKM_CUDA(cudaMemcpyAsync(trace.data(), p.trace, sizeof(int32_t) * rws, cudaMemcpyDeviceToHost, st));
  CKM_CUDA(cudaMemcpyAsync(doms.data(), p.doms, sizeof(DomainOut) * doms.size(), cudaMemcpyDeviceToHost, st));
  CKM_CUDA(cudaStreamSynchronize(st));
  return CKM_OK;
}

static int do_search(ckm_engine *e, const ckm_models *m, const int32_t *model_idx, int32_t nmodels, const int64_t *bin_model_offsets,
                     const ckm_seqdb *db, double Ecut, double domEcut, ckm_hit **hits_out, int64_t *nhits_out);

static int do_align(ckm_engine *e, const ckm_models *m, int32_t model, const ckm_seqdb *db, int32_t *state_out, float *oasc_out) {
  if (!e || !m || !db || !state_out) { set_error("ckm_align: bad argument"); return CKM_EINVAL; }
  if (model < 0 || model >= (int)m->models.size()) { set_error("ckm_align: model index out of range"); return CKM_EINVAL; }
  cudaSetDevice(e->device);
  std::memset(&e->stats, 0, sizeof(e->stats));
  const int nseq = db->nseq;
  for (int64_t i = 0; i < db->nres; ++i) state_out[i] = 0;
  if (oasc_out) for (int s = 0; s < nseq; ++s) oasc_out[s] = 0.0f;
  std::vector<PairWork> pairs;
  std::vector<Envelope> envs;
  int64_t rows = 0;
  auto add = [&](int s, int i, int j) {
    PairWork pw{};
    pw.seq = s; pw.model = model; pw.L = db->len[s]; pw.first_dom = (int32_t)pairs.size(); pw.ndom_slots = 1; pw.row_off = rows;
    rows += pw.L + 1;
    Envelope en{};
    en.pair = (int32_t)pairs.size(); en.i = i; en.j = j; en.null2_done = 1; en.slot = (int32_t)pairs.size();
    pairs.push_back(pw); envs.push_back(en);
  };
  for (int s = 0; s < nseq; ++s) if (db->len[s] > 0) add(s, 1, db->len[s]);
  if (pairs.empty()) return CKM_OK;
  std::vector<int32_t> trace; std::vector<DomainOut> doms;
  int rc;
  if ((rc = align_pass(e, m, db, pairs, envs, rows, trace, doms))) return rc;
  auto emit = [&](const std::vector<PairWork> &pp, const std::vector<DomainOut> &dd, const std::vector<int32_t> &tr, std::vector<int> *failed) {
    for (size_t pi = 0; pi < pp.size(); ++pi) {
      const PairWork &pw = pp[pi];
      if (!dd[pi].ok) { if (failed) failed->push_back(pw.seq); continue; }
      if (oasc_out) oasc_out[pw.seq] = dd[pi].oasc;
      int32_t *dst = state_out + (db->offsets[pw.seq] - db->offsets[0]);
      for (int i = 1; i <= pw.L; ++i) dst[i - 1] = tr[pw.row_off + i];
    }
  };
  std::vector<int> failed;
  emit(pairs, doms, trace, &failed);
  if (failed.empty()) return CKM_OK;
  // the rare sequences one unihit envelope cannot hold: the envelope of the best domain the search pipeline defines
  ckm_hit *hits = nullptr; int64_t nhits = 0;
  if ((rc = do_search(e, m, &model, 1, nullptr, db, 1e300, 1e300, &hits, &nhits))) return rc;
  std::vector<int> best(nseq, -1);
  for (int64_t h = 0; h < nhits; ++h) { const int s = hits[h].seq; if (best[s] < 0 || hits[h].dom_score > hits[best[s]].dom_score) best[s] = (int)h; }
  pairs.clear(); envs.clear(); rows = 0;
  for (int s : failed) if (best[s] >= 0) add(s, hits[best[s]].env_from, hits[best[s]].env_to);
  std::free(hits);
  if (pairs.empty()) return CKM_OK;
  if ((rc = align_pass(e, m, db, pairs, envs, rows, trace, doms))) return rc;
  emit(pairs, doms, trace, nullptr);
  return CKM_OK;
}

}  // namespace ckm

extern "C" int ckm_align(ckm_engine *e, const ckm_models *m, int32_t model, const ckm_seqdb *db, int32_t *state_out, float *oasc_out) {
  return ckm::do_align(e, m, model, db, state_out, oasc_out);
}
