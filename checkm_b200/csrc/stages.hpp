// stages.hpp -- parameter blocks and launchers of the device stages (kernels_*.cu), shared with search.cu.
#pragma once
#include "engine.hpp"

namespace ckm {

#ifndef CKM_SSV_WARPS
#define CKM_SSV_WARPS 16
#endif
constexpr int SSV_WARPS = CKM_SSV_WARPS;
constexpr int SSV_WARPS_HOST = SSV_WARPS;
constexpr int MSV_WARPS = 8;

// ---- stage 1a: SSV pre-filter over all (ORF x HMM) pairs ----
struct SsvParams {
  const uint8_t *res; const int64_t *off; const int32_t *len; const int32_t *bin;
  const float *msvB; const int32_t *tjb; const int32_t *order;
  int32_t nseq, seq_chunk, nchunks;
  const TileGroup *groups; const int32_t *group_list; int32_t ngroups;
  const TileDesc *tiles; const TileModel *tile_models;
  const int32_t *chain_first_tile, *chain_ntiles;
  const uint8_t *tile_blob;
  const uint8_t *tile_active;      // [nbins][ntiles] or null
  const uint8_t *model_active;     // [nbins][nmodels] or null
  int32_t ntiles, nmodels;
  int32_t *unit_counter;
  int2 *cand; int32_t *cand_count; int32_t cand_cap;
  int16_t *bnd; int64_t bnd_stride;   // per-warp boundary columns for chained tiles (2 buffers of bnd_stride each)
  unsigned long long *cells;          // statistics: DP cells swept
  // Resolving a pair in the SSV epilogue: while the J state cannot have fired (u_max below the J bound and the int8 cap) the
  // maximum of the sweep IS the MSV filter's xE, so the exact score and its P-value follow from u_max alone and the pair goes
  // straight to the pass list; only J-eligible / capped / chained pairs are forwarded to the exact MSV kernels.
  int32_t resolve;                    // 1: resolve in the epilogue (CKM_SSV_RESOLVE=0 forwards every firing pair, as a cross-check)
  const ModelScalars *ms; const float *nullsc;
  Candidate *pass; int32_t *pass_count; int32_t pass_cap;
  int32_t *resolved_count;            // pairs scored here (statistics)
  int32_t *xj_dense; const int32_t *model_slot;   // parity output (see MsvParams)
  double F1;
};

int launch_ssv(int J, bool tmem, const SsvParams &p, int grid, size_t smem_bytes, cudaStream_t stream);   // tmem: J = 32 tiles in the TMEM-assisted layout

// ---- stage 1b: exact MSV on the candidates ----
struct MsvParams {
  const uint8_t *res; const int64_t *off; const int32_t *len;
  const float *nullsc; const int32_t *tjb;
  const ModelScalars *ms; const uint8_t *rbv; const uint32_t *rmb;
  const int2 *cand; const int32_t *cand_count; int32_t cand_cap;
  Candidate *out; int32_t *out_count; int32_t out_cap;
  int32_t *xj_dense;           // optional [nmodel_slots][nseq] dense output for parity tests (null in production)
  const int32_t *model_slot;   // database model index -> row of xj_dense
  int32_t nseq;
  int32_t row_bytes;           // shared-memory bytes of one DP row (>= maxM+2)
  int32_t use_blk;             // 1: models with msv2_ok go to the lane-blocked kernels, 0: every candidate to msv_exact_kernel
  double F1;
};

int launch_msv_exact(const MsvParams &p, int grid, cudaStream_t stream);           // models without a lane-block class
// every (sequence, model) pair of the models that have no SSV tiles, appended to the candidate list of the exact kernels
int launch_ssv_bypass(const int32_t *models, int32_t nbypass, int32_t nseq, const int32_t *len, const int32_t *bin,
                      const uint8_t *model_active, int32_t nmodels_db, int2 *cand, int32_t *cand_count, int32_t cand_cap,
                      cudaStream_t stream);
int launch_msv2(const MsvParams &p, int cls, int grid, cudaStream_t stream);       // lane-blocked, class index 0..9

// ---- stages 2-4: bias filter, ViterbiFilter, ForwardParser on the survivors ----
constexpr int VIT_WARPS = 4;
constexpr int FWD_WARPS = 4;
struct FilterParams {
  const uint8_t *res; const int64_t *off; const int32_t *len;
  const float *lenA, *lenB;          // L*log(p1), log(1-p1) of each sequence (host-computed, libm-exact)
  const int16_t *tmove_w;
  const ModelScalars *ms;
  const float *bias_eo; const int16_t *rwv; const int16_t *twv; const float *rfv; const float *tfv;
  const uint4 *twb; const uint32_t *rwb; const float4 *tfb; const float *rfb;   // lane-blocked tables
  const uint4 *twp; const uint32_t *rwp;                                         // packed Viterbi tables
  Candidate *redo; int32_t *redo_count; int32_t redo_cap;                       // pairs the packed Viterbi kernel hands to the int32 kernels
  int32_t *vit_work;                 // N_BLK_CLASSES zeroed cursors into `in`, one per packed-Viterbi class kernel (null: static strides)
  const Candidate *in; const int32_t *in_count; int32_t in_cap;
  Candidate *out; int32_t *out_count; int32_t out_cap;
  int32_t row_elems;                 // shared-memory elements of one DP row
  double F1, F2, F3;
  int32_t use_blk;                   // 1: models with a blocked class go to the *2 kernels
  // optional dense outputs for parity tests
  float *dense_filtersc, *dense_vit, *dense_fwd; uint8_t *dense_passed;
  const int32_t *model_slot; int32_t nseq;
};
int launch_bias(const FilterParams &p, int grid, cudaStream_t st);
int launch_vit(const FilterParams &p, int grid, cudaStream_t st);
// lane-block classes: class index c (0..9) keeps BLK_Q[c] model positions per lane; index 10 = the unblocked kernels
constexpr int N_BLK_CLASSES = 10;
constexpr int BLK_Q[N_BLK_CLASSES] = {2, 4, 6, 8, 12, 16, 20, 24, 28, 32};
int launch_vit2(const FilterParams &p, int cls, int grid, cudaStream_t st);
int launch_vitp(const FilterParams &p, int cls, int grid, cudaStream_t st);   // packed int16x2 kernels (kernels_vitp.cu)
int launch_all_pairs(Candidate *out, int32_t *count, const int32_t *slot_model, int32_t nslots, int32_t nseq, cudaStream_t st);
int launch_fwd(const FilterParams &p, int grid, cudaStream_t st);

// ---- stage 5: domain definition ----
#define FLT_MIN_F 1.17549435e-38f
struct PairWork {          // one pair that passed the Forward filter
  int32_t seq, model, L;
  int32_t first_dom, ndom_slots;     // its envelopes/domains occupy doms[first_dom .. first_dom+ndom_slots)
  float   fwdsc, filtersc, usc;
  int64_t row_off;                   // offset (in rows of L+1) of its per-residue arrays
};
struct Region { int32_t pair, i, j, multi; };
constexpr int ENS_MAXENV = 32;      // envelopes (= domain slots) a multi-domain region can yield before its capacities are raised
// capacities of one multi-domain region in the trace ensemble (kernels_ensemble.cu); the defaults, raised on demand
struct EnsembleCaps { int32_t segments, trace_segments, envelopes; };
constexpr EnsembleCaps ENS_DEFAULT_CAPS = {4096, 64, ENS_MAXENV};
struct Envelope { int32_t pair, i, j, null2_done; int64_t scratch_off; int32_t slot, pad; };   // slot: index of its DomainOut
struct DomainOut {
  int32_t pair, ienv, jenv, hmmfrom, hmmto, sqfrom, sqto, ok;
  float   envsc, domcorrection, oasc, bitscore, dombias, pad;
  double  lnP;
};
struct HitOut { float pre_score, score, sum_score; int32_t ndom, valid, pad; double lnP; };
struct DomdefParams {
  const uint8_t *res; const int64_t *off; const float *nullsc;
  const ModelScalars *ms; const float *rfv; const float *tfv;
  const PairWork *pairs; int32_t npairs;
  const int32_t *pair_order; int32_t pair_begin, pair_end;   // regions kernels walk pair_order[pair_begin..pair_end) (one class, longest first)
  float *xf, *xb, *btot, *etot, *mocc, *n2sc;      // per-pair arrays, indexed by row_off
  int32_t *trace;                                  // optional (ckm_align): state of every residue in the optimal-accuracy trace, indexed like n2sc:
                                                   //   k > 0 match state k, k < 0 insert state -k, 0 outside the aligned region
  Region *regions; int32_t *region_count; int32_t region_cap;
  const Envelope *envs; const int32_t *env_order; int32_t env_begin, env_end;   // envelope kernels walk env_order[env_begin..env_end)
  float *scratch;
  DomainOut *doms; HitOut *hits;
  const float *logsum_tbl;
  int32_t row_elems;
  const float4 *tfb; const float *rfb;   // lane-blocked tables
  int32_t use_blk;                       // 1: models with a blocked class go to the *2 kernels
};
int launch_regions(const DomdefParams &p, int grid, cudaStream_t st);
int launch_envelopes(const DomdefParams &p, int grid, cudaStream_t st);
int launch_scores(const DomdefParams &p, int grid, cudaStream_t st);
int launch_fwd2(const FilterParams &p, int cls, int grid, cudaStream_t st);
int launch_regions2(const DomdefParams &p, int cls, int grid, cudaStream_t st);
int launch_envelopes2(const DomdefParams &p, int cls, int grid, cudaStream_t st);

}  // namespace ckm
