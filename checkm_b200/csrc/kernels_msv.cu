// kernels_msv.cu -- stage 1 of the cascade: the ungapped (SSV) pre-filter over every (ORF x HMM) pair, and the
// exact MSV filter for the few pairs it forwards.  Replaces the MSV stage of the hmmsearch process CheckM spawns
// (checkm/hmmer.py:70-71); >97% of all DP cells of a search are scored here.
//
// Arithmetic (bit-exact with the 8-bit MSV definition, SURVEY.md A.5 step 1).  The MSV cell update is
//     sv(i,k) = sat0( min255( max(sv(i-1,k-1), xB) + bias ) - cost_k(x_i) )
// With the J state idle, xB is the constant xB0 = base - tjb(L) - tbm(M), and w = max(sv, xB0) obeys
//     w(i,k) = max( w(i-1,k-1) + (bias - cost), xB0 ).
// We carry u = w - xB0 >= 0 in int16 lanes: u' = max(u + d, 0) with d = bias - cost -- ONE DPX instruction
// (VIADDMNMX.S16x2) for two cells, and the running row maximum is folded two words at a time (VIMNMX3.S16x2).
// The J state can only matter once some xE exceeds base + tec, so any pair whose u_max reaches either that bound
// or (conservatively) the filter's pass threshold is re-scored by the exact byte-for-byte MSV kernel below; all
// other pairs are provably rejected by the real filter.  No value ever has to be exact once it is past the bound,
// so int16 wrap-around after thousands of rows is harmless (the maximum was recorded before the wrap).
#include <algorithm>
#include "engine.hpp"
#include "device_utils.cuh"
#include "stages.hpp"

namespace ckm {

// ------------------------------------------------------------------------------------------------
// SSV pre-filter
// ------------------------------------------------------------------------------------------------

template <int J, bool TM> __host__ __device__ constexpr int tile_table_bytes() { return ssv_table_bytes(J, TM); }
template <int J, bool TM> __host__ __device__ constexpr int tile_block_bytes() { return ssv_block_bytes(J, TM); }
constexpr uint32_t SSV_TMEM_COLS = 512;   // a TMEM-assisted CTA owns all of the SM's tensor memory (one CTA per SM)

// TM: words 0..SSV_TMEM_WORDS-1 of every row come from tensor memory at column x * SSV_TMEM_WORDS of lane tmem_lane
template <int J, bool TM>
__device__ __forceinline__ void ssv_rows(const uint8_t *__restrict__ res, int L, uint32_t tile_smem, uint32_t tmem_lane, int lane,
                                         uint32_t sel, const int16_t *bnd_in, int16_t *bnd_out, uint32_t (&u)[J], uint32_t &xE) {
  constexpr int G = J / 4;
  const uint4 *rp = reinterpret_cast<const uint4 *>(res);
  const uint32_t lane_off = tile_smem + lane * 16;
  constexpr bool I8 = ssv_int8_chunk(J, TM);          // words 0..7 of every lane come as int8 pairs in one 16-byte chunk
  constexpr int G0 = I8 ? SSV_I8_WORDS / 4 : TM ? SSV_TMEM_WORDS / 4 : 0;       // int16 quads read from shared memory start here
  static_assert(!TM || J == 32, "TMEM-assisted tiles are J = 32 tiles");
  auto do_row = [&](uint32_t x, int i) {
    const uint32_t row = lane_off + x * ssv_row_bytes(J, TM);
    uint4 e[G];
    uint32_t t[TM ? SSV_TMEM_WORDS : 1];
    if constexpr (TM) tmem_ld16(tmem_lane + x * SSV_TMEM_WORDS, t);
    if (I8) {
      const uint4 c = lds128(row);
      const uint32_t cw[4] = {c.x, c.y, c.z, c.w};
#pragma unroll
      for (int q = 0; q < SSV_I8_WORDS; ++q) (&e[q >> 2].x)[q & 3] = prmt_b32(cw[q >> 1], 0u, (q & 1) ? 0xB3A2u : 0x9180u);   // sign-extend a byte pair
    }
#pragma unroll
    for (int g = G0; g < G; ++g) e[g] = lds128(row + (g - (I8 ? G0 - 1 : 0)) * 512);
    if constexpr (TM) {
      tmem_wait_ld(t);
#pragma unroll
      for (int q = 0; q < SSV_TMEM_WORDS; ++q) (&e[q >> 2].x)[q & 3] = t[q];
    }
    uint32_t bndw = 0;
    if (bnd_in != nullptr) bndw = (i > 0) ? (uint32_t)(uint16_t)bnd_in[i - 1] : 0u;      // chained tile: cell 0 continues the previous chunk's last cell
    const uint32_t sh = __shfl_sync(0xffffffffu, u[J - 1], (lane + 31) & 31);
#pragma unroll
    for (int q = J - 1; q >= 1; --q) {
      const uint32_t d = (&e[q >> 2].x)[q & 3];
      u[q] = __viaddmax_s16x2_relu(u[q - 1], d, 0x80008000u);     // max(u + d, 0): the relu form takes its floor as an immediate (a literal 0 operand costs a register zeroing per use)
    }
    const uint32_t p0 = __byte_perm(sh, bndw, sel);
    u[0] = __viaddmax_s16x2_relu(p0, e[0].x, 0x80008000u);
#pragma unroll
    for (int q = 0; q < J; q += 2) xE = __vimax3_s16x2(xE, u[q], u[q + 1]);
    if (bnd_out != nullptr && lane == 31) bnd_out[i] = (int16_t)(u[J - 1] >> 16);
  };
  // full blocks of 16 rows, then the tail in groups of 4 (at most 3 padding rows are swept; they score -inf everywhere)
  const int nfull = L >> 4;
  uint4 cur = __ldg(rp);
  for (int b = 0; b < nfull; ++b) {
    const uint4 nxt = __ldg(rp + b + 1);          // the stream is padded to a multiple of 16 and the next ORF (or the buffer's slack) follows
    const uint32_t w4[4] = {cur.x, cur.y, cur.z, cur.w};
#pragma unroll
    for (int r = 0; r < 16; ++r) do_row((w4[r >> 2] >> (8 * (r & 3))) & 0xffu, b * 16 + r);
    cur = nxt;
  }
  const int ntail = ((L & 15) + 3) >> 2;
  for (int t = 0; t < ntail; ++t) {
    const uint32_t w = (t == 0) ? cur.x : (t == 1) ? cur.y : (t == 2) ? cur.z : cur.w;
#pragma unroll
    for (int r = 0; r < 4; ++r) do_row((w >> (8 * r)) & 0xffu, nfull * 16 + t * 4 + r);
  }
}

// TM: a TMEM-assisted J = 32 tile (every group holds one tile, models.cu).  Warp w reads the tensor-memory lanes of its
// sub-partition, 32 * (w % 4) + lane, so each of the four lane quarters holds its own copy of the tile's TMEM words.
template <int J, bool TM>
__global__ void __launch_bounds__(SSV_WARPS * 32, 1) ssv_kernel(SsvParams p) {
  static_assert(!TM || SSV_WARPS % 4 == 0, "every sub-partition needs warps to fill its copy of the TMEM words");
  extern __shared__ __align__(128) uint8_t smem[];
  __shared__ __align__(8) uint64_t bar;
  __shared__ int s_unit, s_item;
  __shared__ uint32_t s_tmem;
  __shared__ int16_t su[SSV_WARPS][64];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const uint32_t smem_base = smem_u32(smem);
  const uint32_t sel = (lane == 0) ? 0x1054u : 0x3210u;
  constexpr int TB = tile_block_bytes<J, TM>();
  // gains clamped to int8 are exact only while u < 128, so a slot that reaches 127 is flagged as a candidate
  constexpr int I8CAP = ssv_int8_chunk(J, TM) ? 127 : 32767;
  if (warp == 0) {
    if (TM) tmem_alloc(&s_tmem, SSV_TMEM_COLS);
    if (lane == 0) { mbar_init(&bar, 1); fence_mbar_init(); }
  }
  if (TM) tmem_fence_before_sync();
  __syncthreads();
  if (TM) tmem_fence_after_sync();
  const uint32_t tmem_lane = TM ? s_tmem + ((uint32_t)(32 * (warp & 3)) << 16) : 0u;
  uint32_t phase = 0;
  int cur_group = -1;
  unsigned long long my_cells = 0;
  int16_t *bndA = p.bnd ? p.bnd + ((int64_t)(blockIdx.x * SSV_WARPS + warp) * 2) * p.bnd_stride : nullptr;
  int16_t *bndB = p.bnd ? bndA + p.bnd_stride : nullptr;

  while (true) {
    if (TM) tmem_fence_before_sync();
    __syncthreads();                       // everybody is done with the previous unit (tables + s_item)
    if (TM) tmem_fence_after_sync();
    if (tid == 0) { s_unit = atomicAdd(p.unit_counter, 1); s_item = 0; }
    __syncthreads();
    const int unit = s_unit;
    if (unit >= p.ngroups * p.nchunks) break;
    const int gi = unit / p.nchunks, chunk = unit % p.nchunks;
    const TileGroup grp = p.groups[p.group_list[gi]];
    if (gi != cur_group) {                 // stage this group's tables (TMA bulk copies, one per tile)
      cur_group = gi;
      if (tid == 0) {
        fence_proxy_async();
        mbar_expect_tx(&bar, (uint32_t)grp.table_bytes);
        for (int t = 0; t < grp.ntiles; ++t)
          bulk_g2s(smem_base + t * TB, p.tile_blob + grp.table_off + (int64_t)t * TB, TB, &bar);
      }
      mbar_wait(&bar, phase);
      phase ^= 1;
      if constexpr (TM) {                  // copy words 0..SSV_TMEM_WORDS-1 of every row into this sub-partition's TMEM lanes
        for (int x = warp >> 2; x < KPAD; x += SSV_WARPS / 4) {
          const uint32_t row = smem_base + lane * 16 + x * ssv_row_bytes(J, TM);
          uint32_t w[SSV_TMEM_WORDS];
#pragma unroll
          for (int g = 0; g < SSV_TMEM_WORDS / 4; ++g) {
            const uint4 v = lds128(row + g * 512);
            w[4 * g] = v.x; w[4 * g + 1] = v.y; w[4 * g + 2] = v.z; w[4 * g + 3] = v.w;
          }
          tmem_st16(tmem_lane + x * SSV_TMEM_WORDS, w);
        }
        tmem_wait_st();
        tmem_fence_before_sync();
        __syncthreads();
        tmem_fence_after_sync();
      }
    }
    const int s_begin = chunk * p.seq_chunk;
    const int s_count = min(p.seq_chunk, p.nseq - s_begin);
    const int nitems = s_count * grp.nchains;
    while (true) {
      int it = 0;
      if (lane == 0) it = atomicAdd(&s_item, 1);
      it = __shfl_sync(0xffffffffu, it, 0);
      if (it >= nitems) break;
      const int s = p.order[s_begin + it / grp.nchains];
      const int chain = grp.first_chain + it % grp.nchains;
      const int L = p.len[s];
      if (L == 0) continue;
      const int t0 = p.chain_first_tile[chain], nt = TM ? 1 : p.chain_ntiles[chain];     // J = 32 tiles are never chained
      const int sbin = p.bin[s];
      if (p.tile_active != nullptr && !p.tile_active[(int64_t)sbin * p.ntiles + t0]) continue;
      const uint8_t *res = p.res + p.off[s];
      const float Bs = p.msvB[s];
      const int tjb = p.tjb[s];
      bool chain_cand = false;
      for (int tt = 0; tt < nt; ++tt) {
        const int t = t0 + tt;
        const int tl = t - grp.first_tile;                   // tile slot in shared memory
        const uint32_t tsm = smem_base + tl * TB;
        uint32_t u[J];
#pragma unroll
        for (int q = 0; q < J; ++q) u[q] = 0u;
        uint32_t xE = 0u;
        const int16_t *bin_ = (nt > 1 && tt > 0) ? ((tt & 1) ? bndA : bndB) : nullptr;
        int16_t *bout = (nt > 1 && tt + 1 < nt) ? ((tt & 1) ? bndB : bndA) : nullptr;
        ssv_rows<J, TM>(res, L, tsm, tmem_lane, lane, sel, bin_, bout, u, xE);
        my_cells += (unsigned long long)L * (2 * J);
        // ---- epilogue: does any slot reach the candidate bound? ----
        const uint8_t *meta = smem + tl * TB + tile_table_bytes<J, TM>();
        const float *A = reinterpret_cast<const float *>(meta);
        const int32_t *F = reinterpret_cast<const int32_t *>(meta + 256);
        const int32_t *SM = reinterpret_cast<const int32_t *>(meta + 512);
        const int ulo = (int)(int16_t)(xE & 0xffffu), uhi = (int)(int16_t)(xE >> 16);
        const int thr_lo = min(min((int)floorf(A[lane] + Bs) - 1, F[lane] + tjb), I8CAP);
        const int thr_hi = min(min((int)floorf(A[32 + lane] + Bs) - 1, F[32 + lane] + tjb), I8CAP);
        const bool c_lo = (SM[lane] >= 0) && (ulo >= thr_lo);
        const bool c_hi = (SM[32 + lane] >= 0) && (uhi >= thr_hi);
        const unsigned m_lo = __ballot_sync(0xffffffffu, c_lo), m_hi = __ballot_sync(0xffffffffu, c_hi);
        if ((m_lo | m_hi) == 0u) continue;
        if (nt > 1) { chain_cand = true; continue; }
        // which models of the tile own a firing slot?  lane j < nmodels answers for tile model j
        su[warp][lane] = (int16_t)ulo; su[warp][32 + lane] = (int16_t)uhi;      // the 64 slot maxima, for the per-model maximum
        __syncwarp();
        const TileDesc td = p.tiles[t];
        if (lane < td.nmodels) {
          const TileModel tm = p.tile_models[td.first_model + lane];
          const unsigned long long mask = ((unsigned long long)m_hi << 32) | m_lo;
          const unsigned long long range = ((tm.nslots >= 64) ? ~0ull : ((1ull << tm.nslots) - 1ull)) << tm.slot0;
          bool act = (mask & range) != 0ull;
          if (act && p.model_active != nullptr) act = p.model_active[(int64_t)sbin * p.nmodels + tm.model] != 0;
          if (act) {
            int umax = 0;
            for (int z = tm.slot0; z < tm.slot0 + tm.nslots; ++z) umax = max(umax, (int)su[warp][z]);
            const int jbound = min(F[tm.slot0] + tjb, I8CAP);                    // from here on J (or the int8 clamp) could have mattered
            if (!p.resolve || umax >= jbound || umax < 1) {
              const int pos = atomicAdd(p.cand_count, 1);
              if (pos < p.cand_cap) p.cand[pos] = make_int2(s, tm.model);
            } else {
              // exact MSV score: xE_max = u_max + xB0 (u = max(sv, xB0) - xB0 and u_max >= 1), xJ = max(xE_max - tec, 0)
              const ModelScalars ms = p.ms[tm.model];
              const int tjbm = min(tjb + (int)ms.tbm_b, 255);
              const int xB0 = max((int)ms.base_b - tjbm, 0);
              const int xJ = max(umax + xB0 - (int)ms.tec_b, 0);
              float usc = ((float)(xJ - tjb) - (float)ms.base_b);
              usc = __fdiv_rn(usc, ms.scale_b);
              usc = __fsub_rn(usc, 3.0f);
              if (p.xj_dense != nullptr) p.xj_dense[(int64_t)p.model_slot[tm.model] * p.nseq + s] = xJ;
              const float nullsc = p.nullsc[s];
              const float seq_score = __fdiv_rn(__fsub_rn(usc, nullsc), 0.69314718055994529f);
              const double P = gumbel_surv((double)seq_score, (double)ms.evparam[0], (double)ms.evparam[1]);
              atomicAdd(p.resolved_count, 1);
              if (P <= p.F1) {
                const int pos = atomicAdd(p.pass_count, 1);
                if (pos < p.pass_cap) {
                  Candidate cd;
                  cd.seq = s; cd.model = tm.model; cd.usc = usc; cd.filtersc = nullsc; cd.vitsc = 0.f; cd.fwdsc = 0.f; cd.P = P;
                  p.pass[pos] = cd;
                }
              }
            }
          }
        }
        __syncwarp();
      }
      if (nt > 1 && chain_cand && lane == 0) {
        const TileModel tm = p.tile_models[p.tiles[t0].first_model];
        bool act = true;
        if (p.model_active != nullptr) act = p.model_active[(int64_t)sbin * p.nmodels + tm.model] != 0;
        if (act) {
          const int pos = atomicAdd(p.cand_count, 1);
          if (pos < p.cand_cap) p.cand[pos] = make_int2(s, tm.model);
        }
      }
    }
  }
  if (TM && warp == 0) tmem_release(s_tmem, SSV_TMEM_COLS);     // the loop's last barrier ordered every warp's TMEM reads before this
  // statistics
  my_cells = warp_sum_ull(my_cells);
  if (lane == 0 && p.cells != nullptr) atomicAdd(p.cells, my_cells);
}

template __global__ void ssv_kernel<4, false>(SsvParams);
template __global__ void ssv_kernel<8, false>(SsvParams);
template __global__ void ssv_kernel<16, false>(SsvParams);
template __global__ void ssv_kernel<32, false>(SsvParams);
template __global__ void ssv_kernel<32, true>(SsvParams);

template <int J, bool TM>
static int launch_ssv_t(const SsvParams &p, int grid, size_t smem_bytes, cudaStream_t stream) {
  cudaError_t e = cudaFuncSetAttribute(ssv_kernel<J, TM>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes);
  if (e != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute(ssv_kernel)");
  ssv_kernel<J, TM><<<grid, SSV_WARPS * 32, smem_bytes, stream>>>(p);
  e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail(e, "ssv_kernel launch");
  return CKM_OK;
}

int launch_ssv(int J, bool tmem, const SsvParams &p, int grid, size_t smem_bytes, cudaStream_t stream) {
  switch (J) {
    case 4: return launch_ssv_t<4, false>(p, grid, smem_bytes, stream);
    case 8: return launch_ssv_t<8, false>(p, grid, smem_bytes, stream);
    case 16: return launch_ssv_t<16, false>(p, grid, smem_bytes, stream);
    case 32: return tmem ? launch_ssv_t<32, true>(p, grid, smem_bytes, stream) : launch_ssv_t<32, false>(p, grid, smem_bytes, stream);
    default: set_error("unsupported tile width"); return CKM_EINVAL;
  }
}

// ------------------------------------------------------------------------------------------------
// Exact MSV filter: one warp per candidate pair, byte-for-byte the 8-bit recurrence with the J state.
// Lane l owns model positions k = l+1, l+33, ...; the previous row lives in shared memory.
// ------------------------------------------------------------------------------------------------


__global__ void __launch_bounds__(MSV_WARPS * 32) msv_exact_kernel(MsvParams p) {
  extern __shared__ __align__(128) uint8_t smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint8_t *row0 = smem + (size_t)warp * 2 * p.row_bytes, *row1 = row0 + p.row_bytes;
  const int ncand = min(*p.cand_count, p.cand_cap);
  for (int c = blockIdx.x * MSV_WARPS + warp; c < ncand; c += gridDim.x * MSV_WARPS) {
    const int2 pr = p.cand[c];
    const int s = pr.x, m = pr.y;
    const ModelScalars ms = p.ms[m];
    if (p.use_blk && ms.msv2_ok) continue;  // handled by msv2_kernel<Q> (CKM_BLK=0 sends every model here)
    const int M = ms.M, L = p.len[s];
    const uint8_t *res = p.res + p.off[s];
    const uint8_t *rbv = p.rbv + (int64_t)ms.off_cells * KPAD;
    const int tjb = p.tjb[s];
    const int tjbm = min(tjb + (int)ms.tbm_b, 255);
    const int bias = ms.bias_b, base = ms.base_b, tec = ms.tec_b;
    for (int k = lane; k <= M + 1; k += 32) { row0[k] = 0; row1[k] = 0; }
    __syncwarp();
    int xJ = 0, xB = max(base - tjbm, 0);
    bool overflow = false;
    uint8_t *prev = row0, *cur = row1;
    for (int i = 0; i < L; ++i) {
      const int x = res[i];
      const uint8_t *rsc = rbv + (int64_t)x * ms.Mpad;
      int xE = 0;
      for (int k = lane + 1; k <= M; k += 32) {
        int sv = max((int)prev[k - 1], xB);
        sv = min(sv + bias, 255);
        sv = max(sv - (int)rsc[k], 0);
        cur[k] = (uint8_t)sv;
        xE = max(xE, sv);
      }
      xE = warp_max_int(xE);
      if (min(xE + bias, 255) == 255) { overflow = true; break; }
      xE = max(xE - tec, 0);
      xJ = max(xJ, xE);
      xB = max(max(base, xJ) - tjbm, 0);
      __syncwarp();
      uint8_t *tmp = prev; prev = cur; cur = tmp;
    }
    __syncwarp();
    if (lane == 0) {
      float usc;
      if (overflow) usc = INFINITY;
      else {
        usc = ((float)(xJ - tjb) - (float)base);
        usc = __fdiv_rn(usc, ms.scale_b);
        usc = __fsub_rn(usc, 3.0f);
      }
      if (p.xj_dense != nullptr) p.xj_dense[(int64_t)p.model_slot[m] * p.nseq + s] = overflow ? 256 : xJ;
      const float nullsc = p.nullsc[s];
      const float seq_score = __fdiv_rn(__fsub_rn(usc, nullsc), 0.69314718055994529f);
      const double P = gumbel_surv((double)seq_score, (double)ms.evparam[0], (double)ms.evparam[1]);
      if (P <= p.F1) {
        const int pos = atomicAdd(p.out_count, 1);
        if (pos < p.out_cap) {
          Candidate cd;
          cd.seq = s; cd.model = m; cd.usc = usc; cd.filtersc = nullsc; cd.vitsc = 0.f; cd.fwdsc = 0.f; cd.P = P;
          p.out[pos] = cd;
        }
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Exact MSV, lane-blocked: lane l keeps model positions l*Q+1 .. l*Q+Q of the row in Q/2 registers of two int16
// (word j = positions j and Q/2+j of the block, so the k-1 dependency is a register rename plus one shuffle and one
// byte permute per row).  The byte recurrence  sv = sat0(sat255(max(sv', xB) + bias) - cost)  is evaluated as
// max(max(sv', xB) + (bias - cost), 0): the 255 clamp cannot fire before the row-level overflow test does (every
// operand is <= the previous row's xE or xB, both < 255 - bias; models with base + bias >= 255 stay on the byte kernel),
// so the bytes are those of msv_exact_kernel.  2 packed instructions per 2 cells instead of ~8 scalar ones per cell.
// ------------------------------------------------------------------------------------------------
template <int Q>
__global__ void __launch_bounds__(128) msv2_kernel(MsvParams p) {
  constexpr int H = Q / 2;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, wpb = blockDim.x >> 5;
  const int ncand = min(*p.cand_count, p.cand_cap);
  for (int c = blockIdx.x * wpb + warp; c < ncand; c += gridDim.x * wpb) {
    const int2 pr = p.cand[c];
    const int s = pr.x, m = pr.y;
    const ModelScalars ms = p.ms[m];
    if (ms.vq != Q || !ms.msv2_ok) continue;
    const int L = p.len[s];
    const uint32_t *rmb = p.rmb + ms.blk_off * 32 * (KPAD / 2) + lane;
    const int tjb = p.tjb[s];
    const int tjbm = min(tjb + (int)ms.tbm_b, 255);
    const int bias = ms.bias_b, base = ms.base_b, tec = ms.tec_b;
    // The registers hold u = max(sv, xB) - xB >= 0 (as the SSV pre-filter does), so a row is u' = max(u + gain, 0): one
    // VIADDMNMX.RELU per word instead of a max with xB and an add.  max_k u' + xB = max(xE, xB), and using that in place of
    // xE changes neither the xB trajectory (it can only lift an xJ that is still below base, which xB ignores) nor the final
    // xJ as long as some cell of the pair was positive (then the best row has xE > xB).  When xB moves by delta, u is
    // re-based: u <- max(u - delta, 0).  A pair without a single positive cell falls back to the plain recurrence.
    uint32_t sv[H];
#pragma unroll
    for (int j = 0; j < H; ++j) sv[j] = 0u;
    int xJ = 0, xB = max(base - tjbm, 0);
    bool overflow = false;
    int umax = 0;
    const uint4 *rp = reinterpret_cast<const uint4 *>(p.res + p.off[s]);
    const int nblk = (L + 15) >> 4;
    auto row = [&](const uint32_t (&e)[H]) -> uint32_t {
      uint32_t up = __shfl_up_sync(0xffffffffu, sv[H - 1], 1);
      if (lane == 0) up = 0u;
      const uint32_t in0 = __byte_perm(up, sv[H - 1], 0x5432);     // lo: position below my block, hi: my position Q/2
#pragma unroll
      for (int j = H - 1; j >= 1; --j) sv[j] = __viaddmax_s16x2_relu(sv[j - 1], e[j], 0x80008000u);
      sv[0] = __viaddmax_s16x2_relu(in0, e[0], 0x80008000u);
      uint32_t xEv = sv[0];
      if (H == 1) { }
      else if (H & 1) {
#pragma unroll
        for (int j = 1; j + 1 < H; j += 2) xEv = __vimax3_s16x2(xEv, sv[j], sv[j + 1]);
      } else {
        xEv = __vmaxs2(xEv, sv[1]);
#pragma unroll
        for (int j = 2; j + 1 < H; j += 2) xEv = __vimax3_s16x2(xEv, sv[j], sv[j + 1]);
      }
      return xEv;
    };
    // Rows go in groups of four with ONE warp reduction per group: xB = max(base, xJ) - tjbm moves only when some row's
    // xE - tec exceeds max(base, xJ), and while it does not, xJ after the group is max(xJ, group max - tec) -- exactly what the
    // row-by-row recurrence gives.  A group whose maximum could move xB (or overflow) is replayed row by row from the saved
    // registers; that happens only around the few high-scoring rows of a pair.
    uint4 r16 = (nblk > 0) ? __ldg(rp) : make_uint4(0, 0, 0, 0);
    for (int b = 0; b < nblk && !overflow; ++b) {
      const uint4 rnext = (b + 1 < nblk) ? __ldg(rp + b + 1) : make_uint4(0, 0, 0, 0);
      for (int j4 = 0; j4 < 4 && !overflow; ++j4) {
        const int i0 = b * 16 + j4 * 4;
        if (i0 >= L) break;
        const uint32_t wcur = (j4 == 0) ? r16.x : (j4 == 1) ? r16.y : (j4 == 2) ? r16.z : r16.w;
        const int nrow = min(4, L - i0);
        uint32_t eg[4][H];
#pragma unroll
        for (int rr = 0; rr < 4; ++rr) {
          const uint32_t x = (wcur >> (8 * rr)) & 0xffu;       // rows past L read the padding code: a valid table row, never used
#pragma unroll
          for (int j = 0; j < H; ++j) eg[rr][j] = __ldg(rmb + (x * H + j) * 32);
        }
        uint32_t cp[H];
#pragma unroll
        for (int j = 0; j < H; ++j) cp[j] = sv[j];
        uint32_t xEg = 0u;
#pragma unroll
        for (int rr = 0; rr < 4; ++rr) if (rr < nrow) xEg = __vmaxs2(xEg, row(eg[rr]));
        int uE = max((int)(xEg & 0xffffu), (int)(xEg >> 16));
        uE = __reduce_max_sync(0xffffffffu, uE);
        const int xE = uE + xB;                               // = max(row maxima of sv, xB)
        if (xE + bias < 255 && xE - tec <= max(base, xJ)) {
          xJ = max(xJ, max(xE - tec, 0));
          umax = max(umax, uE);
        } else {
#pragma unroll
          for (int j = 0; j < H; ++j) sv[j] = cp[j];
#pragma unroll
          for (int rr = 0; rr < 4; ++rr) {
            if (rr < nrow && !overflow) {
              const uint32_t xEv = row(eg[rr]);
              int ue = max((int)(xEv & 0xffffu), (int)(xEv >> 16));
              ue = __reduce_max_sync(0xffffffffu, ue);
              umax = max(umax, ue);
              int xe = ue + xB;
              if (xe + bias >= 255) overflow = true;
              else {
                xe = max(xe - tec, 0);
                xJ = max(xJ, xe);
                const int xBn = max(max(base, xJ) - tjbm, 0);
                if (xBn != xB) {                              // re-base u on the new xB (xB never decreases)
                  const uint32_t nd = (uint32_t)(uint16_t)(int16_t)(xB - xBn) * 0x00010001u;
#pragma unroll
                  for (int j = 0; j < H; ++j) sv[j] = __viaddmax_s16x2_relu(sv[j], nd, 0x80008000u);
                  xB = xBn;
                }
              }
            }
          }
        }
      }
      r16 = rnext;
    }
    if (!overflow && umax == 0) {
      // no positive cell anywhere (never the case for a pair the SSV pre-filter forwards on a positive threshold): the plain
      // recurrence, row by row, with the exact row maxima of sv
      xJ = 0; xB = max(base - tjbm, 0);
#pragma unroll
      for (int j = 0; j < H; ++j) sv[j] = 0u;
      for (int i = 0; i < L && !overflow; ++i) {
        const uint32_t x = p.res[p.off[s] + i];
        uint32_t e[H];
#pragma unroll
        for (int j = 0; j < H; ++j) e[j] = __ldg(rmb + (x * H + j) * 32);
        const uint32_t XBw = (uint32_t)xB * 0x00010001u;
        uint32_t up = __shfl_up_sync(0xffffffffu, sv[H - 1], 1);
        if (lane == 0) up = 0u;
        const uint32_t in0 = __byte_perm(up, sv[H - 1], 0x5432);
        uint32_t xEv = 0u;
#pragma unroll
        for (int j = H - 1; j >= 1; --j) { sv[j] = __viaddmax_s16x2_relu(__vmaxs2(sv[j - 1], XBw), e[j], 0x80008000u); xEv = __vmaxs2(xEv, sv[j]); }
        sv[0] = __viaddmax_s16x2_relu(__vmaxs2(in0, XBw), e[0], 0x80008000u);
        xEv = __vmaxs2(xEv, sv[0]);
        int xe = max((int)(xEv & 0xffffu), (int)(xEv >> 16));
        xe = __reduce_max_sync(0xffffffffu, xe);
        if (xe + bias >= 255) overflow = true;
        else { xe = max(xe - tec, 0); xJ = max(xJ, xe); xB = max(max(base, xJ) - tjbm, 0); }
      }
    }
    if (lane == 0) {
      float usc;
      if (overflow) usc = INFINITY;
      else {
        usc = ((float)(xJ - tjb) - (float)base);
        usc = __fdiv_rn(usc, ms.scale_b);
        usc = __fsub_rn(usc, 3.0f);
      }
      if (p.xj_dense != nullptr) p.xj_dense[(int64_t)p.model_slot[m] * p.nseq + s] = overflow ? 256 : xJ;
      const float nullsc = p.nullsc[s];
      const float seq_score = __fdiv_rn(__fsub_rn(usc, nullsc), 0.69314718055994529f);
      const double P = gumbel_surv((double)seq_score, (double)ms.evparam[0], (double)ms.evparam[1]);
      if (P <= p.F1) {
        const int pos = atomicAdd(p.out_count, 1);
        if (pos < p.out_cap) {
          Candidate cd;
          cd.seq = s; cd.model = m; cd.usc = usc; cd.filtersc = nullsc; cd.vitsc = 0.f; cd.fwdsc = 0.f; cd.P = P;
          p.out[pos] = cd;
        }
      }
    }
  }
}

int launch_msv2(const MsvParams &p, int cls, int grid, cudaStream_t stream) {
  switch (cls) {
    case 0: msv2_kernel<2><<<grid, 128, 0, stream>>>(p); break;
    case 1: msv2_kernel<4><<<grid, 128, 0, stream>>>(p); break;
    case 2: msv2_kernel<6><<<grid, 128, 0, stream>>>(p); break;
    case 3: msv2_kernel<8><<<grid, 128, 0, stream>>>(p); break;
    case 4: msv2_kernel<12><<<grid, 128, 0, stream>>>(p); break;
    case 5: msv2_kernel<16><<<grid, 128, 0, stream>>>(p); break;
    case 6: msv2_kernel<20><<<grid, 128, 0, stream>>>(p); break;
    case 7: msv2_kernel<24><<<grid, 128, 0, stream>>>(p); break;
    case 8: msv2_kernel<28><<<grid, 128, 0, stream>>>(p); break;
    case 9: msv2_kernel<32><<<grid, 128, 0, stream>>>(p); break;
    default: set_error("launch_msv2: bad class"); return CKM_EINVAL;
  }
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? CKM_OK : cuda_fail(e, "msv2_kernel launch");
}

// Models too long for a chain of SSV tiles (models.cu: ssv_bypass) skip the pre-filter: all of their pairs become candidates.
__global__ void ssv_bypass_kernel(const int32_t *models, int32_t nbypass, int32_t nseq, const int32_t *len, const int32_t *bin,
                                  const uint8_t *model_active, int32_t nmodels_db, int2 *cand, int32_t *cand_count, int32_t cand_cap) {
  const int64_t n = (int64_t)nbypass * nseq;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int s = (int)(i % nseq), m = models[i / nseq];
    if (len[s] == 0) continue;
    if (model_active != nullptr && !model_active[(int64_t)bin[s] * nmodels_db + m]) continue;
    const int pos = atomicAdd(cand_count, 1);
    if (pos < cand_cap) cand[pos] = make_int2(s, m);
  }
}

int launch_ssv_bypass(const int32_t *models, int32_t nbypass, int32_t nseq, const int32_t *len, const int32_t *bin,
                      const uint8_t *model_active, int32_t nmodels_db, int2 *cand, int32_t *cand_count, int32_t cand_cap,
                      cudaStream_t stream) {
  if (nbypass <= 0 || nseq <= 0) return CKM_OK;
  const int64_t n = (int64_t)nbypass * nseq;
  const int grid = (int)std::min<int64_t>(1184, (n + 255) / 256);
  ssv_bypass_kernel<<<grid, 256, 0, stream>>>(models, nbypass, nseq, len, bin, model_active, nmodels_db, cand, cand_count, cand_cap);
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? CKM_OK : cuda_fail(e, "ssv_bypass_kernel launch");
}

int launch_msv_exact(const MsvParams &p, int grid, cudaStream_t stream) {
  const size_t smem = (size_t)MSV_WARPS * 2 * p.row_bytes;
  cudaError_t e = cudaFuncSetAttribute(msv_exact_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute(msv_exact)");
  msv_exact_kernel<<<grid, MSV_WARPS * 32, smem, stream>>>(p);
  e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail(e, "msv_exact_kernel launch");
  return CKM_OK;
}

}  // namespace ckm
