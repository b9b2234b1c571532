// models.cu -- model database on the device: per-model score tables for the survivor stages and the packed SSV tiles.
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <stdexcept>
#include "engine.hpp"

namespace ckm {

static thread_local std::string g_error;
void set_error(const std::string &msg) { g_error = msg; }
const std::string &get_error() { return g_error; }
int cuda_fail(cudaError_t e, const char *what) {
  set_error(std::string("CUDA error: ") + cudaGetErrorString(e) + " in " + what);
  return CKM_ECUDA;
}

static const double kLog2 = 0.69314718055994529;

template <class T>
static int upload(T **dptr, const std::vector<T> &h) {
  size_t bytes = std::max<size_t>(h.size() * sizeof(T), 16);
  CKM_CUDA(cudaMalloc((void **)dptr, bytes));
  if (!h.empty()) CKM_CUDA(cudaMemcpy(*dptr, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice));
  return CKM_OK;
}

// Packs the models into SSV tiles (see engine.hpp) and builds the int16 emission-delta tables.
static void build_tiles(ckm_models &db, std::vector<uint8_t> &blob) {
  const int n = (int)db.models.size();
  struct Item { int model, M; };
  // tile width policy: CKM_SSV_J = auto (4/8/16 by model length) | 8 | 16 | 32 (one width for every model)
  const char *pol = std::getenv("CKM_SSV_J");
  int fixedJ = 32;
  if (pol != nullptr) { if (!std::strcmp(pol, "auto")) fixedJ = 0; else fixedJ = std::atoi(pol); }
  if (fixedJ != 0 && fixedJ != 4 && fixedJ != 8 && fixedJ != 16 && fixedJ != 32) fixedJ = 32;
  // J = 32 table layout: TMEM-assisted (default) or with the int8 chunk (CKM_SSV_TMEM=0, kept as the cross-check)
  { const char *v = std::getenv("CKM_SSV_TMEM"); db.ssv_tmem = !(v != nullptr && v[0] == '0'); }
  const bool tmem = db.ssv_tmem;
  std::vector<Item> cls[3], longm;
  int Js[3] = {4, 8, 16};
  int chainJ = 16;
  if (fixedJ != 0) { Js[0] = Js[1] = Js[2] = fixedJ; chainJ = (fixedJ == 32) ? 16 : fixedJ; }   // chains must fit shared memory together
  for (int i = 0; i < n; ++i) {
    int M = db.models[i].M;
    if (fixedJ != 0) { if (M <= 64 * fixedJ - 1) cls[0].push_back({i, M}); else longm.push_back({i, M}); }
    else if (M <= 255) cls[0].push_back({i, M});
    else if (M <= 511) cls[1].push_back({i, M});
    else if (M <= 1023) cls[2].push_back({i, M});
    else longm.push_back({i, M});
  }
  struct HostTile { int J; std::vector<TileModel> tm; int used; int chain_prev, chain_next; };
  std::vector<HostTile> tiles;
  std::vector<std::pair<int, int>> chains;   // (first tile, ntiles)
  std::vector<int> tile_class;
  for (int c = 0; c < 3; ++c) {
    auto &v = cls[c];
    std::stable_sort(v.begin(), v.end(), [](const Item &a, const Item &b) { return a.M > b.M; });
    const int J = Js[c];
    size_t first = tiles.size();
    for (const Item &it : v) {
      int W = it.M / J + 1;
      size_t t;
      for (t = first; t < tiles.size(); ++t)
        if (tiles[t].used + W <= 64 && (int)tiles[t].tm.size() < 32) break;
      if (t == tiles.size()) { tiles.push_back({J, {}, 0, 0, 0}); tile_class.push_back(c); }
      tiles[t].tm.push_back({it.model, tiles[t].used, W, 0});
      tiles[t].used += W;
    }
    for (size_t t = first; t < tiles.size(); ++t) chains.push_back({(int)t, 1});
  }
  const int chunk_cells = 64 * chainJ;
  const int64_t cap = 200000;                 // shared-memory budget of one tile group
  db.ssv_bypass.clear();
  for (const Item &it : longm) {
    int ncells = it.M + 1;                    // real cells + the mandatory padding cell
    int nch = (ncells + chunk_cells - 1) / chunk_cells;
    // All chunks of a chain sit in shared memory together.  A model whose chain does not fit (M >= 3072) gets no tiles:
    // every pair of it goes straight to the exact MSV kernel (ssv_bypass_kernel), which has no such limit.
    if ((int64_t)nch * ssv_block_bytes(chainJ, tmem) > cap) { db.ssv_bypass.push_back(it.model); continue; }
    chains.push_back({(int)tiles.size(), nch});
    for (int c = 0; c < nch; ++c) {
      HostTile ht{chainJ, {}, 64, c > 0, c + 1 < nch};
      ht.tm.push_back({it.model, 0, 64, c});
      tiles.push_back(ht);
      tile_class.push_back(3);
    }
  }
  // groups: consecutive chains of equal J up to the shared-memory budget
  db.tiles.clear(); db.tile_models.clear(); db.groups.clear(); db.chain_first_tile.clear(); db.chain_ntiles.clear();
  int64_t off = 0;
  for (size_t t = 0; t < tiles.size(); ++t) {
    TileDesc td{};
    td.J = tiles[t].J; td.first_model = (int)db.tile_models.size(); td.nmodels = (int)tiles[t].tm.size();
    td.chain_next = tiles[t].chain_next; td.chain_prev = tiles[t].chain_prev; td.table_off = off;
    for (auto &tm : tiles[t].tm) db.tile_models.push_back(tm);
    db.tiles.push_back(td);
    off += ssv_block_bytes(td.J, tmem);
  }
  blob.assign((size_t)off, 0);
  {
    TileGroup g{}; bool open = false; int64_t gbytes = 0;
    for (size_t c = 0; c < chains.size(); ++c) {
      int t0 = chains[c].first, nt = chains[c].second, J = tiles[t0].J;
      int64_t need = (int64_t)nt * ssv_block_bytes(J, tmem);
      if (need > cap) throw std::runtime_error("model " + db.models[tiles[t0].tm[0].model].name + " is too long for the SSV tiles");
      // a TMEM-assisted tile is alone in its group: tensor memory holds the words of one tile
      if (open && (g.J != J || gbytes + need > cap || (tmem && J == 32))) { g.table_bytes = gbytes; db.groups.push_back(g); open = false; }
      if (!open) { g = TileGroup{}; g.J = J; g.first_tile = t0; g.ntiles = 0; g.nchains = 0; g.first_chain = (int)c; g.table_off = db.tiles[t0].table_off; gbytes = 0; open = true; }
      g.ntiles += nt; g.nchains += 1; gbytes += need;
      db.chain_first_tile.push_back(t0); db.chain_ntiles.push_back(nt);
    }
    if (open) { g.table_bytes = gbytes; db.groups.push_back(g); }
  }
  // tables
  for (size_t t = 0; t < tiles.size(); ++t) {
    const int J = tiles[t].J;
    uint8_t *base = blob.data() + db.tiles[t].table_off;
    const bool i8 = ssv_int8_chunk(J, tmem);
    const int RB = ssv_row_bytes(J, tmem);
    float *A = reinterpret_cast<float *>(base + ssv_table_bytes(J, tmem));
    int32_t *F = reinterpret_cast<int32_t *>(base + ssv_table_bytes(J, tmem) + 256);
    int32_t *SM = reinterpret_cast<int32_t *>(base + ssv_table_bytes(J, tmem) + 512);
    for (int s = 0; s < 64; ++s) { A[s] = 1e30f; F[s] = 1 << 28; SM[s] = -1; }
    // where the gain of cell (lane, half, q) for residue x lives, and a store that knows the cell's width
    auto put = [&](int x, int lane, int half, int q, int d) {
      uint8_t *row = base + (size_t)x * RB;
      if (i8 && q < SSV_I8_WORDS) reinterpret_cast<int8_t *>(row)[lane * 16 + 2 * q + half] = (int8_t)std::max(d, -128);
      else {
        const int g = (q >> 2) - (i8 ? (SSV_I8_WORDS / 4 - 1) : 0);      // 16-byte chunk index inside the row
        reinterpret_cast<int16_t *>(row + ((size_t)g * 32 + lane) * 16)[(q & 3) * 2 + half] = (int16_t)std::max(d, -32768);
      }
    };
    // default: padding everywhere
    for (int x = 0; x < KPAD; ++x) for (int lane = 0; lane < 32; ++lane) for (int half = 0; half < 2; ++half) for (int q = 0; q < J; ++q) put(x, lane, half, q, -32768);
    for (size_t j = 0; j < tiles[t].tm.size(); ++j) {
      const TileModel &tm = tiles[t].tm[j];
      const Model &m = db.models[tm.model];
      const int W1 = m.M + 1;
      for (int sl = 0; sl < tm.nslots; ++sl) {
        const int slot = tm.slot0 + sl;
        A[slot] = db.models[tm.model].M > 0 ? 0.0f : 0.0f;   // filled below
        SM[slot] = (int)j;
        const int lane = slot & 31, half = slot >> 5;
        for (int q = 0; q < J; ++q) {
          const int k = tm.chunk * 64 * J + sl * J + q + 1;    // model position of this cell
          if (k > m.M) continue;
          for (int x = 0; x < KP; ++x) {
            put(x, lane, half, q, (int)m.bias_b - (int)m.rbv[(size_t)x * W1 + k]);
          }
        }
      }
    }
  }
  // thresholds (per slot) need the per-model A, F
  for (size_t t = 0; t < tiles.size(); ++t) {
    const int J = tiles[t].J;
    uint8_t *base = blob.data() + db.tiles[t].table_off;
    float *A = reinterpret_cast<float *>(base + ssv_table_bytes(J, tmem));
    int32_t *F = reinterpret_cast<int32_t *>(base + ssv_table_bytes(J, tmem) + 256);
    for (auto &tm : tiles[t].tm) {
      const Model &m = db.models[tm.model];
      const double F1 = 0.02;
      const double sstar = (double)m.evparam[0] - std::log(-std::log(1.0 - F1)) / (double)m.evparam[1];
      const float Am = (float)((double)m.tbm_b + (double)m.tec_b + (double)m.scale_b * kLog2 * sstar);
      for (int sl = 0; sl < tm.nslots; ++sl) { A[tm.slot0 + sl] = Am; F[tm.slot0 + sl] = 4 + (int)m.tbm_b; }
    }
  }
}

int models_build_device(ckm_models &db) {
  const int n = (int)db.models.size();
  std::vector<ModelScalars> sc(n);
  int64_t cols = 0, blk_units = 0;
  db.maxM = 0;
  for (int i = 0; i < n; ++i) {
    const Model &m = db.models[i];
    ModelScalars &s = sc[i];
    std::memset(&s, 0, sizeof(s));
    s.M = m.M; s.Mpad = ((m.M + 1) + 31) / 32 * 32 + 32; s.off_cells = (int32_t)cols;
    cols += s.Mpad;
    s.tbm_b = m.tbm_b; s.tec_b = m.tec_b; s.base_b = m.base_b; s.bias_b = m.bias_b;
    s.base_w = m.base_w; s.xw_e_loop = m.xw_e_loop; s.xw_e_move = m.xw_e_move;
    s.scale_b = m.scale_b; s.scale_w = m.scale_w;
    for (int z = 0; z < 6; ++z) s.evparam[z] = m.evparam[z];
    s.ddbound_w = m.ddbound_w;
    {
      int emax = 0, tbm = 0;
      for (int x = 0; x < KP; ++x) for (int k = 1; k <= m.M; ++k) emax = std::max(emax, (int)m.rwv[(size_t)x * (m.M + 1) + k]);
      for (int k = 1; k <= m.M; ++k) tbm = std::min(tbm, (int)m.twv[(size_t)k * T_N + 0]);
      s.vit_emax = (int16_t)emax; s.vit_tbm = (int16_t)tbm;
    }
    s.vq = (m.M <= 64) ? 2 : (m.M <= 128) ? 4 : (m.M <= 192) ? 6 : (m.M <= 256) ? 8 : (m.M <= 384) ? 12 : (m.M <= 512) ? 16 : (m.M <= 640) ? 20 : (m.M <= 768) ? 24 : (m.M <= 896) ? 28 : (m.M <= 1024) ? 32 : 0;
    s.blk_off = blk_units;
    s.msv2_ok = (s.vq != 0 && (int)m.base_b + (int)m.bias_b < 255) ? 1 : 0;
    blk_units += s.vq;
    db.maxM = std::max(db.maxM, m.M);
    if (m.M > MAX_MODEL_M) {
      set_error("model " + m.name + " has " + std::to_string(m.M) + " positions; the engine's DP rows hold at most " + std::to_string(MAX_MODEL_M));
      return CKM_EINVAL;
    }
  }
  if (cols > (int64_t)1 << 30) { set_error("model database too large"); return CKM_ENOMEM; }
  db.total_cols = cols;
  std::vector<uint8_t> rbv((size_t)cols * KPAD, 255);
  std::vector<int16_t> rwv((size_t)cols * KPAD, -32768), twv((size_t)cols * T_N, -32768);
  std::vector<float> rfv((size_t)cols * KPAD, 0.0f), tfv((size_t)cols * T_N, 0.0f), beo((size_t)n * KPAD * 2, 1.0f);
  for (int i = 0; i < n; ++i) {
    const Model &m = db.models[i];
    const ModelScalars &s = sc[i];
    const size_t W1 = (size_t)m.M + 1;
    for (int x = 0; x < KP; ++x)
      for (int k = 0; k <= m.M; ++k) {
        const size_t d = ((size_t)s.off_cells * KPAD) + (size_t)x * s.Mpad + k;
        rbv[d] = m.rbv[x * W1 + k]; rwv[d] = m.rwv[x * W1 + k]; rfv[d] = m.rfv[x * W1 + k];
      }
    for (int k = 0; k <= m.M; ++k)
      for (int z = 0; z < T_N; ++z) {
        twv[((size_t)s.off_cells + k) * T_N + z] = m.twv[(size_t)k * T_N + z];
        tfv[((size_t)s.off_cells + k) * T_N + z] = m.tfv[(size_t)k * T_N + z];
      }
    for (int x = 0; x < KP; ++x) { beo[((size_t)i * KPAD + x) * 2] = m.bias_eo[x][0]; beo[((size_t)i * KPAD + x) * 2 + 1] = m.bias_eo[x][1]; }
  }
  // lane-blocked tables
  std::vector<uint4> twb((size_t)std::max<int64_t>(blk_units, 1) * 32);
  std::vector<uint32_t> rwb((size_t)std::max<int64_t>(blk_units, 1) * 32 * KPAD / 2 + 32);
  std::vector<uint32_t> rmb((size_t)std::max<int64_t>(blk_units, 1) * 32 * KPAD / 2 + 32);
  std::vector<float4> tfb((size_t)std::max<int64_t>(blk_units, 1) * 32 * 2);
  std::vector<uint4> twp((size_t)std::max<int64_t>(blk_units, 1) * 32);              // W = vq/2 words x 32 lanes x 2 uint4
  std::vector<uint32_t> rwp((size_t)std::max<int64_t>(blk_units, 1) * 32 * KPAD / 2 + 32);
  std::vector<float> rfb((size_t)std::max<int64_t>(blk_units, 1) * 32 * KPAD);
  for (int i = 0; i < n; ++i) {
    const Model &m = db.models[i];
    const ModelScalars &s = sc[i];
    const int Q = s.vq;
    if (Q == 0) continue;
    const size_t W1 = (size_t)m.M + 1;
    for (int q = 0; q < Q; ++q)
      for (int lane = 0; lane < 32; ++lane) {
        const int k = lane * Q + q + 1;
        int16_t tw[8]; float tf[8];
        for (int z = 0; z < 8; ++z) { tw[z] = (k <= m.M) ? m.twv[(size_t)k * T_N + z] : (int16_t)-32768; tf[z] = (k <= m.M) ? m.tfv[(size_t)k * T_N + z] : 0.0f; }
        uint4 u;
        u.x = (uint16_t)tw[0] | ((uint32_t)(uint16_t)tw[1] << 16); u.y = (uint16_t)tw[2] | ((uint32_t)(uint16_t)tw[3] << 16);
        u.z = (uint16_t)tw[4] | ((uint32_t)(uint16_t)tw[5] << 16); u.w = (uint16_t)tw[6] | ((uint32_t)(uint16_t)tw[7] << 16);
        twb[((size_t)s.blk_off + q) * 32 + lane] = u;
        tfb[(((size_t)s.blk_off + q) * 32 + lane) * 2] = make_float4(tf[0], tf[1], tf[2], tf[3]);
        tfb[(((size_t)s.blk_off + q) * 32 + lane) * 2 + 1] = make_float4(tf[4], tf[5], tf[6], tf[7]);
        for (int x = 0; x < KPAD; ++x) {
          const int16_t ew = (k <= m.M && x < KP) ? m.rwv[(size_t)x * W1 + k] : (int16_t)-32768;
          const float ef = (k <= m.M && x < KP) ? m.rfv[(size_t)x * W1 + k] : 0.0f;
          // emissions of a model: [x][Q/2][32] words at (blk_off*32*KPAD/2) ; floats [x][Q][32] at blk_off*32*KPAD
          uint32_t &w = rwb[(size_t)s.blk_off * 32 * KPAD / 2 + ((size_t)x * (Q / 2) + (q >> 1)) * 32 + lane];
          if (q & 1) w = (w & 0x0000ffffu) | ((uint32_t)(uint16_t)ew << 16); else w = (w & 0xffff0000u) | (uint16_t)ew;
          rfb[(size_t)s.blk_off * 32 * KPAD + ((size_t)x * Q + q) * 32 + lane] = ef;
          // MSV gains bias - cost; word j of a lane pairs its positions j and Q/2 + j, so a one-position shift stays
          // inside the register file.  Positions past M can never score.
          const int cost = (k <= m.M && x < KP) ? (int)m.rbv[(size_t)x * W1 + k] : 255;
          const int16_t eg = (k <= m.M) ? (int16_t)((int)m.bias_b - cost) : (int16_t)-20000;
          uint32_t &wm = rmb[(size_t)s.blk_off * 32 * KPAD / 2 + ((size_t)x * (Q / 2) + (q % (Q / 2))) * 32 + lane];
          if (q >= Q / 2) wm = (wm & 0x0000ffffu) | ((uint32_t)(uint16_t)eg << 16); else wm = (wm & 0xffff0000u) | (uint16_t)eg;
        }
      }
  }
  // packed Viterbi tables (kernels_vitp.cu): entries clamped at -22528 and values floored at -10240, so no int16 add can wrap
  for (int i = 0; i < n; ++i) {
    const Model &m = db.models[i];
    const ModelScalars &s = sc[i];
    if (s.vq == 0) continue;
    const int W = s.vq / 2;
    const size_t W1 = (size_t)m.M + 1;
    auto clampw = [](int v) { return (uint32_t)(uint16_t)(int16_t)std::max(v, -22528); };
    for (int w = 0; w < W; ++w)
      for (int lane = 0; lane < 32; ++lane) {
        const int k0 = lane * W + w + 1, k1 = 32 * W + k0;
        uint32_t tw[8];
        for (int z = 0; z < 8; ++z) {
          const int a = (k0 <= m.M) ? (int)m.twv[(size_t)k0 * T_N + z] : -32768, b = (k1 <= m.M) ? (int)m.twv[(size_t)k1 * T_N + z] : -32768;
          tw[z] = clampw(a) | (clampw(b) << 16);
        }
        const size_t base = ((size_t)s.blk_off / 2 * 32 + (size_t)w * 32 + lane) * 2;
        twp[base] = make_uint4(tw[0], tw[1], tw[2], tw[3]);
        twp[base + 1] = make_uint4(tw[4], tw[5], tw[6], tw[7]);
        for (int x = 0; x < KPAD; ++x) {
          const int a = (k0 <= m.M && x < KP) ? (int)m.rwv[(size_t)x * W1 + k0] : -32768, b = (k1 <= m.M && x < KP) ? (int)m.rwv[(size_t)x * W1 + k1] : -32768;
          rwp[(size_t)s.blk_off * 32 * KPAD / 2 + ((size_t)x * W + w) * 32 + lane] = clampw(a) | (clampw(b) << 16);
        }
      }
  }
  int st;
  if ((st = upload(&db.d_twp, twp))) return st;
  if ((st = upload(&db.d_rwp, rwp))) return st;
  if ((st = upload(&db.d_twb, twb))) return st;
  if ((st = upload(&db.d_rwb, rwb))) return st;
  if ((st = upload(&db.d_rmb, rmb))) return st;
  if ((st = upload(&db.d_tfb, tfb))) return st;
  if ((st = upload(&db.d_rfb, rfb))) return st;
  if ((st = upload(&db.d_scalars, sc))) return st;
  if ((st = upload(&db.d_rbv, rbv))) return st;
  if ((st = upload(&db.d_rwv, rwv))) return st;
  if ((st = upload(&db.d_twv, twv))) return st;
  if ((st = upload(&db.d_rfv, rfv))) return st;
  if ((st = upload(&db.d_tfv, tfv))) return st;
  if ((st = upload(&db.d_bias_eo, beo))) return st;
  std::vector<uint8_t> blob;
  try { build_tiles(db, blob); } catch (const std::exception &ex) { set_error(ex.what()); return CKM_EINVAL; }
  db.tile_blob_bytes = (int64_t)blob.size();
  if ((st = upload(&db.d_tile_blob, blob))) return st;
  if ((st = upload(&db.d_tiles, db.tiles))) return st;
  if ((st = upload(&db.d_tile_models, db.tile_models))) return st;
  if ((st = upload(&db.d_groups, db.groups))) return st;
  if ((st = upload(&db.d_chain_first_tile, db.chain_first_tile))) return st;
  if ((st = upload(&db.d_chain_ntiles, db.chain_ntiles))) return st;
  if ((st = upload(&db.d_ssv_bypass, db.ssv_bypass))) return st;
  return CKM_OK;
}

void models_free_device(ckm_models &db) {
  cudaFree(db.d_scalars); cudaFree(db.d_rbv); cudaFree(db.d_rwv); cudaFree(db.d_twv); cudaFree(db.d_rfv); cudaFree(db.d_tfv);
  cudaFree(db.d_bias_eo); cudaFree(db.d_twb); cudaFree(db.d_twp); cudaFree(db.d_rwp); cudaFree(db.d_rwb); cudaFree(db.d_rmb); cudaFree(db.d_tfb); cudaFree(db.d_rfb); cudaFree(db.d_tile_blob); cudaFree(db.d_tiles); cudaFree(db.d_tile_models); cudaFree(db.d_groups);
  cudaFree(db.d_chain_first_tile); cudaFree(db.d_chain_ntiles); cudaFree(db.d_ssv_bypass);
}

}  // namespace ckm
