// engine.hpp -- internal structures of libckm.so (host + device views).  Layout notes are in DESIGN.md.
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <string>
#include <vector>
#include "../../include/ckm.h"
#include "hmm_model.hpp"

namespace ckm {
// Longest model the engine takes.  The chunked fp32 kernels (M > 1024) keep three DP rows of ((M + 31) / 32 * 32 + 64) floats per
// warp, four warps per CTA, in shared memory: 4 * 3 * 4 * (4608 + 64) = 224,256 of the 232,448 bytes a CTA may own.
constexpr int MAX_MODEL_M = 4608;

// ------------------------------------------------------------------------------------------------
// SSV tiles.  A tile is what one warp sweeps down a sequence: 64 "slots" (lane l low half = slot l,
// lane l high half = slot 32+l) x J int16 words per lane.  A model of length M placed at slot s0 with
// W = floor(M/J)+1 slots owns cells k-1 = (slot-s0)*J + q; cells past M are padding (score -32768), and the
// last cell of the last slot is always padding so nothing leaks into the next model of the tile.
// Emission table of a tile in HBM/shared memory: int16 [KPAD residues][J/4 quads][32 lanes][4 q][2 halves]
// i.e. per residue row J*32 32-bit words; lane l reads quad g as one 128-bit load at word (g*32 + l)*4.
// J = 32 tiles keep the first two quads (words 0..7 of every lane) as int8 pairs in ONE 16-byte chunk per lane
// (gains clamped at -128, exact while u < 128; the kernel flags any slot that reaches 127): 7 instead of 8 LDS.128 per
// row, the sign-extending unpack costs one PRMT per word on the ALU pipe, which has the headroom.
// TMEM-assisted J = 32 tiles (the default, ckm_models::ssv_tmem) keep every word as int16 instead: the kernel copies words
// 0..SSV_TMEM_WORDS-1 of every lane and residue into tensor memory once per tile, and a row then reads them with one
// tcgen05.ld next to 4 LDS.128 for the rest (tensor memory feeds registers without using the shared-memory pipe).
// ------------------------------------------------------------------------------------------------
constexpr int SSV_I8_WORDS = 8;       // words per lane stored as int8 pairs in J = 32 tiles without tensor memory
constexpr int SSV_TMEM_WORDS = 16;    // words per lane read from tensor memory in TMEM-assisted J = 32 tiles
static_assert(KPAD * SSV_TMEM_WORDS <= 512, "a TMEM-assisted tile must fit the 512 tensor-memory columns of an SM");
__host__ __device__ constexpr bool ssv_int8_chunk(int J, bool tmem) { return J == 32 && !tmem; }
__host__ __device__ constexpr int ssv_row_bytes(int J, bool tmem) {
  return ssv_int8_chunk(J, tmem) ? 128 * J - 16 * 32 * (SSV_I8_WORDS / 4 - 1) : 128 * J;
}
__host__ __device__ constexpr int ssv_table_bytes(int J, bool tmem) { return KPAD * ssv_row_bytes(J, tmem); }
__host__ __device__ constexpr int ssv_block_bytes(int J, bool tmem) { return ssv_table_bytes(J, tmem) + 768; }
struct TileModel {       // one model (or one 1024-cell chunk of a long model) inside a tile
  int32_t model;         // database index
  int32_t slot0, nslots;
  int32_t chunk;         // chunk number for chained (M >= 1024) models, else 0
};

struct TileDesc {
  int32_t J;             // 4, 8 or 16
  int32_t first_model;   // index into tile_models
  int32_t nmodels;       // models packed into this tile
  int32_t chain_next;    // 1 if the next tile continues the same long model (its boundary column feeds it)
  int32_t chain_prev;    // 1 if this tile continues the previous one
  int32_t pad;
  int64_t table_off;     // byte offset of the tile's emission table in the tile blob
};

struct TileGroup {       // tiles staged into shared memory together (same J)
  int32_t J;
  int32_t first_tile, ntiles;
  int32_t nchains;       // work items per sequence = chains (a chain = 1 tile, or all chunks of one long model)
  int32_t first_chain;   // index into chain_first_tile
  int32_t pad;
  int64_t table_off;     // byte offset of the group's first table (tables of a group are contiguous)
  int64_t table_bytes;
};

// Per-model scalars used by device code.
struct ModelScalars {
  int32_t M;
  int32_t off_cells;     // offset (in table "columns") of this model in the per-model tables; column stride Mpad
  int32_t Mpad;          // (M+1) rounded up to 32
  uint8_t tbm_b, tec_b, base_b, bias_b;
  int16_t base_w, xw_e_loop, xw_e_move;
  int16_t msv2_ok;       // 1: the lane-blocked MSV kernel applies (vq != 0 and base_b + bias_b < 255, so its adds cannot saturate)
  float   scale_b, scale_w;
  float   evparam[6];
  int32_t ddbound_w;     // lazy-F bound of the Viterbi filter
  int16_t vit_emax;      // largest Viterbi emission word of the model (>= 0): packed-kernel values stay < 32767 - vit_emax
  int16_t vit_tbm;       // most negative B->M entry word (<= 0)
  int32_t vq;            // lane-blocked class: cells per lane (2,4,8,16), 0 = model too long for the blocked kernels
  int64_t blk_off;       // offset of the model's lane-blocked tables (in units of 32 lanes x vq cells)
};

struct Candidate {       // an (ORF, HMM) pair moving down the cascade
  int32_t seq, model;
  float   usc;           // MSV score (nats), INFINITY on overflow
  float   filtersc;      // bias-filter null score (nats)
  float   vitsc, fwdsc;
  double  P;             // P-value after the latest stage
};

// Workspace roles: each keys one grow-only device buffer of the engine (pool.hpp).  Buffers that are live at the same time in
// one call never share a key.  Shared between entry points (same role; one engine runs one call at a time): the filter-cascade
// keys by every entry point that runs the cascade, and Pairs, Vec, Doms, EnvScratch, Envs1, EnvOrder1 by search and alignment.
enum class Ws : int {
  ModelSlot, ModelActive, TileActive, Cand, Pass, Cells, Bnd, GroupList, ListA, ListB, Redo,
  SlotModel, DenseFiltersc, DenseVit, DenseFwd, DensePassed, DenseXj,
  Pairs, Xf, Xb, Vec, LogsumTbl, Regions, PairOrder, Doms, Hits, AlignTrace,
  EnvScratch, Envs1, EnvOrder1, Envs2, EnvOrder2,
  EnsRegions, EnsMultiIdx, EnsScratchOff, EnsScratch, EnsEnvs, EnsCount, EnsCaps, EnsEnvOff, EnsNeed,   // the trace ensemble (on `aux`)
  NtBytes, NtRows, NtPieces, NtStats, NtContigScaf, NtContigLen, NtCounters,
  Gather,
  Count
};

}  // namespace ckm

// ------------------------------------------------------------------------------------------------
// Opaque handles of the C ABI
// ------------------------------------------------------------------------------------------------
struct ckm_models {
  std::vector<ckm::Model> models;
  // device copies
  ckm::ModelScalars *d_scalars = nullptr;
  uint8_t  *d_rbv = nullptr;      // [sum Mpad][KPAD]? no: per model [KPAD][Mpad] bytes, at off_cells*KPAD
  int16_t  *d_rwv = nullptr;      // per model [KPAD][Mpad]
  int16_t  *d_twv = nullptr;      // per model [Mpad][8]
  float    *d_rfv = nullptr;      // per model [KPAD][Mpad]
  float    *d_tfv = nullptr;      // per model [Mpad][8]
  float    *d_bias_eo = nullptr;  // per model [KPAD][2]
  // lane-blocked copies for the register-resident survivor kernels: lane l owns positions k = l*vq + q + 1
  uint4    *d_twb = nullptr;      // per model [vq][32] : 8 int16 transitions of cell (q, lane)
  uint32_t *d_rmb = nullptr;      // per model [KPAD][vq/2][32] : two int16 MSV emission gains bias - cost (q = j, vq/2 + j)
  uint32_t *d_rwb = nullptr;      // per model [KPAD][vq/2][32] : two int16 emissions (q = 2j, 2j+1)
  // packed (int16x2) Viterbi tables: word w of lane l pairs positions k = l*W + w + 1 (low half) and 32*W + k (high half),
  // W = vq/2, every entry clamped to >= -22528 (kernels_vitp.cu)
  uint4    *d_twp = nullptr;      // per model [W][32][2] : {BM MM IM DM} {MD MI II DD}, one int16x2 word each
  uint32_t *d_rwp = nullptr;      // per model [KPAD][W][32]
  float4   *d_tfb = nullptr;      // per model [vq][32][2] : 8 fp32 transitions
  float    *d_rfb = nullptr;      // per model [KPAD][vq][32] : fp32 emission odds
  int64_t   total_cols = 0;
  int       maxM = 0;
  // SSV tiles
  std::vector<ckm::TileDesc>  tiles;
  std::vector<ckm::TileModel> tile_models;
  std::vector<ckm::TileGroup> groups;
  std::vector<int32_t>        chain_first_tile;   // per chain
  std::vector<int32_t>        chain_ntiles;
  std::vector<int32_t>        ssv_bypass;         // models without SSV tiles (chain larger than shared memory): all their pairs are MSV candidates
  bool            ssv_tmem = true;                // J = 32 tiles use the TMEM-assisted layout (CKM_SSV_TMEM=0 at load: the int8-chunk layout)
  int32_t        *d_ssv_bypass = nullptr;
  ckm::TileDesc  *d_tiles = nullptr;
  ckm::TileModel *d_tile_models = nullptr;
  ckm::TileGroup *d_groups = nullptr;
  int32_t        *d_chain_first_tile = nullptr, *d_chain_ntiles = nullptr;
  uint8_t        *d_tile_blob = nullptr;          // emission tables of all tiles
  float          *d_tile_A = nullptr;             // per tile 64 floats: model threshold part per slot
  int32_t        *d_tile_F = nullptr;             // per tile 64 ints: 4 + tbm per slot (flag threshold part)
  int32_t        *d_tile_slot_model = nullptr;    // per tile 64 ints: local model index of each slot, -1 = unused
  int64_t         tile_blob_bytes = 0;
  ckm_engine     *engine = nullptr;
};

struct ckm_seqdb {
  int32_t nseq = 0, nbins = 0;
  int64_t nres = 0;               // residues (unpadded)
  int64_t padded_bytes = 0;
  int32_t maxL = 0;
  std::vector<int64_t> offsets;   // host copy, unpadded CSR
  std::vector<int32_t> bin_of_seq, bin_first_seq, bin_nseq;
  std::vector<int32_t> len;
  // device
  uint8_t *d_res = nullptr;       // every sequence starts 16-byte aligned and is padded to a multiple of 16 with CODE_PAD
  int64_t *d_off = nullptr;       // padded start offsets (nseq+1)
  int32_t *d_len = nullptr;
  int32_t *d_bin = nullptr;
  float   *d_nullsc = nullptr;    // null1 score of each sequence
  int32_t *d_tjb = nullptr;       // MSV N/J/C move cost byte of each sequence
  float   *d_msvB = nullptr;      // sequence part of the SSV candidate threshold
  float   *d_lenA = nullptr, *d_lenB = nullptr;   // L*log(p1), log(1-p1)
  int16_t *d_tmove_w = nullptr;   // Viterbi-filter N/J/C move score of each sequence
  int32_t *d_order = nullptr;     // sequence indices sorted by decreasing length (scheduling order)
  int32_t *d_bin_nseq = nullptr;
  ckm_engine *engine = nullptr;
};

struct ckm_engine {
  int device = 0;
  cudaDeviceProp prop;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev[16];
  // one stream per lane-block class (+1 for the unblocked kernels): the per-class launches of a stage run concurrently
  static constexpr int NCLS = 11;
  cudaStream_t cls[NCLS];
  cudaEvent_t cls_ev[NCLS], fan_ev;
  cudaStream_t aux = nullptr;     // the trace-ensemble job of a search runs here, next to the class streams
  ckm_stats stats;
  // device workspaces by role, reused by every later call (pool.hpp)
  struct { void *p = nullptr; size_t bytes = 0; } ws[(int)ckm::Ws::Count];
  int32_t *d_counters = nullptr;   // small array of device counters
};

namespace ckm {
void set_error(const std::string &msg);
int  cuda_fail(cudaError_t e, const char *what);
#define CKM_CUDA(call) do { cudaError_t _e = (call); if (_e != cudaSuccess) return ckm::cuda_fail(_e, #call); } while (0)
}  // namespace ckm
