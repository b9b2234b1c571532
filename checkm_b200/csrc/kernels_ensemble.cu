// kernels_ensemble.cu -- multi-domain regions: Forward matrix of the region (multihit), 200 stochastic tracebacks with a
// fixed-seed generator, per-trace null2 accumulation, single-linkage clustering of the sampled segments into envelopes
// (SURVEY.md A.5 step 5).  One warp per region; the traceback state machine is warp-uniform, with the O(M) pieces
// (E-state choice, null2 from state counts, link tests) spread over the lanes.
#include <algorithm>
#include <vector>
#include "engine.hpp"
#include "device_utils.cuh"
#include "stages.hpp"
#include "fwdback.cuh"
#include "pool.hpp"

namespace ckm {

constexpr int NSAMPLES = 200;
// Per-region capacities (EnsembleCaps, stages.hpp): sampled segments kept for the clustering, segments of one trace,
// envelopes reported.  The defaults cover regions of up to ~20 domains; a region that needs more says how much in
// `need` and the search repeats its domain phase with that region's capacities raised (search.cu).

struct EnsembleParams {
  DomdefParams d;
  const Region *regions; const int32_t *multi_idx; int32_t nmulti;
  const int64_t *scratch_off;         // per multi region, in floats
  float *scratch;
  const EnsembleCaps *caps;           // per multi region
  const int64_t *env_off;             // per multi region: its first slot in env_out
  Envelope *env_out; int32_t *env_count;      // env_count: envelopes written, or -1 when a capacity was exceeded
  int32_t *need;                      // per multi region x 3: sampled segments, most segments in one trace, significant clusters
};

enum { ST_M = 1, ST_D, ST_I, ST_S, ST_N, ST_B, ST_E, ST_C, ST_T, ST_J };

struct Lcg { uint32_t x; };
__device__ __forceinline__ uint32_t mix3(uint32_t a, uint32_t b, uint32_t c) {
  a -= b; a -= c; a ^= (c >> 13);
  b -= c; b -= a; b ^= (a << 8);
  c -= a; c -= b; c ^= (b >> 13);
  a -= b; a -= c; a ^= (c >> 12);
  b -= c; b -= a; b ^= (a << 16);
  c -= a; c -= b; c ^= (b >> 5);
  a -= b; a -= c; a ^= (c >> 3);
  b -= c; b -= a; b ^= (a << 10);
  c -= a; c -= b; c ^= (b >> 15);
  return c;
}
__device__ __forceinline__ double lcg_random(Lcg &r) { r.x *= 69069u; r.x += 1u; return (double)r.x / 4294967296.0; }

__device__ __forceinline__ int fchoose(Lcg &rng, float *pth, int N) {
  float sum = 0.0f;
  for (int i = 0; i < N; ++i) sum = __fadd_rn(sum, pth[i]);
  if (sum != 0.0f) { const float s = (float)(1.0 / (double)sum); for (int i = 0; i < N; ++i) pth[i] = __fmul_rn(pth[i], s); }
  else for (int i = 0; i < N; ++i) pth[i] = __fdiv_rn(1.0f, (float)N);
  const float roll = (float)lcg_random(rng);
  sum = 0.0f;
  for (int i = 0; i < N; ++i) { sum = __fadd_rn(sum, pth[i]); if (roll < sum) return i; }
  int i;
  int guard = 0;
  do { i = (int)(lcg_random(rng) * N); } while (pth[i] == 0.0f && ++guard < 64);
  return i;
}

__device__ __forceinline__ bool sp_link(const int *a, const int *b) {   // {idx,i,j,k,m}
  int nov = min(a[2], b[2]) - max(a[1], b[1]) + 1;
  int n = min(a[2] - a[1] + 1, b[2] - b[1] + 1);
  if ((float)nov / (float)n < 0.8f) return false;
  nov = min(a[4], b[4]) - max(a[3], b[3]);
  n = min(a[4] - a[3] + 1, b[4] - b[3] + 1);
  if ((float)nov / (float)n < 0.8f) return false;
  if (abs((a[1] - a[3]) - (b[1] - b[3])) > 4) return false;
  if (abs((a[2] - a[4]) - (b[2] - b[4])) > 4) return false;
  return true;
}

__global__ void __launch_bounds__(FWD_WARPS * 32) ensemble_kernel(EnsembleParams ep) {
  extern __shared__ __align__(16) uint8_t smem[];
  const DomdefParams &p = ep.d;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float *rowM = reinterpret_cast<float *>(smem) + (size_t)warp * 3 * p.row_elems;
  float *rowI = rowM + p.row_elems, *rowD = rowI + p.row_elems;
  for (int ri = blockIdx.x * FWD_WARPS + warp; ri < ep.nmulti; ri += gridDim.x * FWD_WARPS) {
    const Region reg = ep.regions[ep.multi_idx[ri]];
    const PairWork pw = p.pairs[reg.pair];
    const ModelScalars ms = p.ms[pw.model];
    FwdModel fm;
    fm.M = ms.M; fm.Mpad = ms.Mpad;
    fm.rfv = p.rfv + (int64_t)ms.off_cells * KPAD;
    fm.tfv = reinterpret_cast<const float4 *>(p.tfv + (int64_t)ms.off_cells * T_N);
    const int M = fm.M, Mpad = fm.Mpad, Lr = reg.j - reg.i + 1;
    const int Q = max(2, (M + 3) / 4);
    const uint8_t *res = p.res + p.off[pw.seq] + (reg.i - 1);
    const Specials sp = make_specials(pw.L, true);
    float *F = ep.scratch + ep.scratch_off[ri];
    float *xf = F + (int64_t)(Lr + 1) * 3 * Mpad;
    float *acc = xf + (int64_t)(Lr + 1) * X_NX, *val = acc + (Lr + 1);
    const EnsembleCaps cap = ep.caps[ri];
    const int SPCAP = cap.segments, TRCAP = cap.trace_segments, MAXENV = cap.envelopes;
    int *spb = reinterpret_cast<int *>(val + (Lr + 1));       // SPCAP x 5
    int *label = spb + (int64_t)SPCAP * 5;                   // 3 x SPCAP: available list, stack, cluster assignment
    int *epc = label + (int64_t)3 * SPCAP;                   // max(Lr, M) + 2
    int *segbuf = epc + max(Lr, M) + 2;                      // per-trace segments, right-to-left: TRCAP x 4
    int most_in_trace = 0;
    float *n2sc = p.n2sc + pw.row_off;
    forward_rows<true, true>(fm, res, Lr, sp, rowM, rowI, rowD, lane, xf, F, 0, nullptr);
    for (int pos = lane; pos <= Lr; pos += 32) acc[pos] = 0.0f;
    __syncwarp();
    Lcg rng; rng.x = mix3(42u, 87654321u, 12345678u); if (rng.x == 0) rng.x = 42;
    // generator jump for the run fast paths: lane l sees draw number l+1 from the current state, x -> jA x + jC
    uint32_t jA = 1u, jC = 0u;
    for (int z = 0; z <= lane; ++z) { jC = jC * 69069u + 1u; jA *= 69069u; }
    int nsp = 0;
    float *cm = rowM, *ci = rowI, *null2 = rowD;
    for (int t = 0; t < NSAMPLES; ++t) {
      for (int pos = lane; pos <= Lr; pos += 32) val[pos] = 1.0f;
      __syncwarp();
      int i = Lr, k = 0, s0 = ST_C, s1 = -1;
      int nseg = 0;
      int sqto = 0, hmmto = 0, sqfrom = 0, hmmfrom = 0, ldom = 0;
      bool in_dom = false, failed = false;
      long guard = 0;
      const long gmax = 8L * (Lr + 2) * (M + 2);
      while (s0 != ST_S) {
        if (++guard > gmax) { failed = true; break; }
        float pth[4];
        // ---- run fast paths.  A walk spends most of its steps in M->M diagonals and in C/J self loops; each step
        // costs one draw and depends only on the cell it stands on, so lane l evaluates the step l places ahead
        // (its cell's path odds, normalised and compared with draw l+1 exactly as the single-step code does) and the
        // warp takes the whole leading run in one memory round trip.  Anything unusual falls to the single-step code. ----
        if (s0 == ST_M || s0 == ST_C || s0 == ST_J) {
          const bool isM = (s0 == ST_M);
          const int ii = i - lane, kk = k - lane;
          const bool valid = isM ? (ii >= 1 && kk >= 1) : (ii >= 0);
          float p0 = 0.f, p1 = 0.f, p2 = 0.f, p3 = 0.f;
          if (valid) {
            if (isM) {
              const float *dpp = F + (int64_t)(ii - 1) * 3 * Mpad;
              const float4 t0 = __ldg(fm.tfv + 2 * kk);
              p0 = __fmul_rn(xf[(int64_t)(ii - 1) * X_NX + X_B], t0.x);
              p1 = __fmul_rn(dpp[kk - 1], t0.y);
              p2 = __fmul_rn(dpp[2 * Mpad + kk - 1], t0.z);
              p3 = __fmul_rn(dpp[Mpad + kk - 1], t0.w);
            } else {
              const int XS = (s0 == ST_C) ? X_C : X_J;
              const float tmv = (s0 == ST_C) ? sp.emove : sp.eloop;
              p0 = (ii > 0) ? __fmul_rn(xf[(int64_t)(ii - 1) * X_NX + XS], sp.nloop) : 0.0f;
              p1 = __fmul_rn(__fmul_rn(xf[(int64_t)ii * X_NX + X_E], tmv), xf[(int64_t)ii * X_NX + X_SCALE]);
            }
          }
          const int np = isM ? 4 : 2;
          float sum = __fadd_rn(__fadd_rn(0.0f, p0), p1);
          if (isM) sum = __fadd_rn(__fadd_rn(sum, p2), p3);
          if (sum != 0.0f) { const float sc = (float)(1.0 / (double)sum); p0 = __fmul_rn(p0, sc); p1 = __fmul_rn(p1, sc); p2 = __fmul_rn(p2, sc); p3 = __fmul_rn(p3, sc); }
          else { const float u = __fdiv_rn(1.0f, (float)np); p0 = u; p1 = u; p2 = u; p3 = u; }
          const uint32_t xl = jA * rng.x + jC;
          const float roll = (float)((double)xl / 4294967296.0);
          const float c0 = __fadd_rn(0.0f, p0), c1 = __fadd_rn(c0, p1), c2 = __fadd_rn(c1, p2), c3 = __fadd_rn(c2, p3);
          int choice = -1;
          if (roll < c0) choice = 0; else if (roll < c1) choice = 1; else if (isM && roll < c2) choice = 2; else if (isM && roll < c3) choice = 3;
          const bool okl = valid && choice >= 0;
          const int stay = isM ? 1 : 0;                   // the choice that continues the run
          const unsigned cont = __ballot_sync(0xffffffffu, okl && choice == stay);
          const int nlead = (cont == 0xffffffffu) ? 32 : (__ffs(~cont) - 1);
          const int okf = (nlead < 32) ? __shfl_sync(0xffffffffu, (int)okl, nlead & 31) : 0;
          const int cf = __shfl_sync(0xffffffffu, choice, nlead & 31);
          const int nproc = nlead + (okf ? 1 : 0);
          if (nproc > 0) {
            guard += nproc - 1;
            if (nlead > 0) {
              if (isM) {
                if (in_dom) {
                  if (sqto == 0) sqto = i - 1;
                  if (hmmto == 0) hmmto = k - 1;
                  sqfrom = i - nlead; hmmfrom = k - nlead; ldom += nlead;
                  if (lane < nlead) cm[k - lane - 1] += 1.0f;
                }
                k -= nlead;
              }
              i -= nlead;
            }
            rng.x = __shfl_sync(0xffffffffu, xl, nproc - 1);
            if (!okf) continue;                           // still inside the run: s0 unchanged
            if (isM) { s1 = (cf == 0) ? ST_B : (cf == 2) ? ST_I : ST_D; k--; i--; }
            else s1 = ST_E;
            goto step_done;
          }
        }
        if (s0 == ST_M) {
          const float *dpp = F + (int64_t)(i - 1) * 3 * Mpad;
          const float4 t0 = __ldg(fm.tfv + 2 * k);
          pth[0] = __fmul_rn(xf[(int64_t)(i - 1) * X_NX + X_B], t0.x);
          pth[1] = __fmul_rn(dpp[k - 1], t0.y);
          pth[2] = __fmul_rn(dpp[2 * Mpad + k - 1], t0.z);
          pth[3] = __fmul_rn(dpp[Mpad + k - 1], t0.w);
          const int c = fchoose(rng, pth, 4);
          s1 = (c == 0) ? ST_B : (c == 1) ? ST_M : (c == 2) ? ST_I : ST_D;
          k--; i--;
        } else if (s0 == ST_D) {
          const float *dpc = F + (int64_t)i * 3 * Mpad;
          const float4 t1 = __ldg(fm.tfv + 2 * (k - 1) + 1);
          pth[0] = __fmul_rn(dpc[k - 1], t1.x);
          pth[1] = __fmul_rn(dpc[Mpad + k - 1], t1.w);
          s1 = fchoose(rng, pth, 2) == 0 ? ST_M : ST_D; k--;
        } else if (s0 == ST_I) {
          const float *dpp = F + (int64_t)(i - 1) * 3 * Mpad;
          const float4 t1 = __ldg(fm.tfv + 2 * k + 1);
          pth[0] = __fmul_rn(dpp[k], t1.y);
          pth[1] = __fmul_rn(dpp[2 * Mpad + k], t1.z);
          s1 = fchoose(rng, pth, 2) == 0 ? ST_M : ST_I; i--;
        } else if (s0 == ST_N) {
          i = 0; s1 = ST_S;                               // N loops back to the start without draws or bookkeeping
        } else if (s0 == ST_C) {
          pth[0] = (i > 0) ? __fmul_rn(xf[(int64_t)(i - 1) * X_NX + X_C], sp.nloop) : 0.0f;
          pth[1] = __fmul_rn(__fmul_rn(xf[(int64_t)i * X_NX + X_E], sp.emove), xf[(int64_t)i * X_NX + X_SCALE]);
          s1 = fchoose(rng, pth, 2) == 0 ? ST_C : ST_E;
        } else if (s0 == ST_J) {
          pth[0] = (i > 0) ? __fmul_rn(xf[(int64_t)(i - 1) * X_NX + X_J], sp.nloop) : 0.0f;
          pth[1] = __fmul_rn(__fmul_rn(xf[(int64_t)i * X_NX + X_E], sp.eloop), xf[(int64_t)i * X_NX + X_SCALE]);
          s1 = fchoose(rng, pth, 2) == 0 ? ST_J : ST_E;
        } else if (s0 == ST_B) {
          pth[0] = __fmul_rn(xf[(int64_t)i * X_NX + X_N], sp.nmove);
          pth[1] = __fmul_rn(xf[(int64_t)i * X_NX + X_J], sp.nmove);
          s1 = fchoose(rng, pth, 2) == 0 ? ST_N : ST_J;
        } else if (s0 == ST_E) {
          // choose among all M(i,k), D(i,k) in the striped enumeration order of the SIMD original:
          // entry e = q*8 + r (match, k = r*Q+q+1) or q*8 + 4 + r (delete)
          const float *dpc = F + (int64_t)i * 3 * Mpad;
          const double roll = lcg_random(rng);
          const float norm = (float)(1.0 / (double)xf[(int64_t)i * X_NX + X_E]);
          const int nent = 8 * Q, per = (nent + 31) / 32;
          const int e0 = lane * per, e1 = min(nent, e0 + per);
          double part = 0.0;
          for (int e = e0; e < e1; ++e) {
            const int q = e >> 3, r = e & 3, isd = (e >> 2) & 1, kk = r * Q + q + 1;
            const float v = (kk <= M) ? __fmul_rn(dpc[isd * Mpad + kk], norm) : 0.0f;
            part += (double)v;
          }
          double incl = part;
#pragma unroll
          for (int o = 1; o < 32; o <<= 1) { const double up = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += up; }
          const unsigned hitmask = __ballot_sync(0xffffffffu, roll < incl && e1 > e0);
          int sel = -1;
          if (hitmask != 0u) {
            const int owner = __ffs(hitmask) - 1;
            if (lane == owner) {
              double sum = incl - part;
              for (int e = e0; e < e1; ++e) {
                const int q = e >> 3, r = e & 3, isd = (e >> 2) & 1, kk = r * Q + q + 1;
                const float v = (kk <= M) ? __fmul_rn(dpc[isd * Mpad + kk], norm) : 0.0f;
                sum += (double)v;
                if (roll < sum) { sel = e; break; }
              }
              if (sel < 0) sel = e1 - 1;
            }
            sel = __shfl_sync(0xffffffffu, sel, owner);
          }
          if (sel < 0) { failed = true; break; }
          { const int q = sel >> 3, r = sel & 3, isd = (sel >> 2) & 1; k = r * Q + q + 1; s1 = isd ? ST_D : ST_M; }
          if (k > M) { failed = true; break; }
          // a new domain starts (we walk right to left, so this is its end)
          in_dom = true; sqto = 0; hmmto = 0; sqfrom = 0; hmmfrom = 0; ldom = 0;
          for (int kk = lane; kk <= M; kk += 32) { cm[kk] = 0.0f; ci[kk] = 0.0f; }
          __syncwarp();
        } else { failed = true; break; }
      step_done:
        // bookkeeping for the state just entered (coordinates k, i are those of s1)
        if (in_dom) {
          if (s1 == ST_M) {
            if (sqto == 0) sqto = i;
            if (hmmto == 0) hmmto = k;
            sqfrom = i; hmmfrom = k; ldom++;
            if (lane == 0) cm[k] += 1.0f;
          } else if (s1 == ST_I) {
            ldom++;
            if (lane == 0) ci[k] += 1.0f;
          } else if (s1 == ST_D) {
            if (hmmto == 0) hmmto = k;
            hmmfrom = k;
          } else if (s1 == ST_B) {
            // domain complete: null2 from its state usage, then the per-residue ratios of the aligned span
            __syncwarp();
            const float nrm = __fdiv_rn(1.0f, (float)ldom);
            for (int kk = lane + 1; kk <= M; kk += 32) { cm[kk] *= nrm; ci[kk] *= nrm; }
            __syncwarp();
            for (int x = 0; x < K; ++x) {
              const float *rp = fm.rfv + (int64_t)x * Mpad;
              float part = 0.0f;
              for (int kk = lane + 1; kk <= M; kk += 32) { part += cm[kk] * __ldg(rp + kk); part += ci[kk]; }
              part = warp_sum_float(part);
              if (lane == 0) null2[x] = part;
            }
            __syncwarp();
            if (lane == 0) {
              { float r = 0.f; r += null2[2]; r += null2[11]; null2[21] = __fdiv_rn(r, 2.0f); }
              { float r = 0.f; r += null2[7]; r += null2[9];  null2[22] = __fdiv_rn(r, 2.0f); }
              { float r = 0.f; r += null2[3]; r += null2[13]; null2[23] = __fdiv_rn(r, 2.0f); }
              null2[24] = null2[8]; null2[25] = null2[1];
              float rx = 0.f;
              for (int x = 0; x < K; ++x) rx += null2[x];
              null2[26] = __fdiv_rn(rx, 20.0f);
              null2[20] = 1.0f; null2[27] = 1.0f; null2[28] = 1.0f; null2[29] = 1.0f;
            }
            __syncwarp();
            // residues sqfrom+1 .. sqto get the ratio; sqfrom itself keeps 1.0 (as the reference does)
            for (int pos = sqfrom + 1 + lane; pos <= sqto; pos += 32) val[pos] = null2[res[pos - 1]];
            if (lane == 0 && nseg < TRCAP) { segbuf[nseg * 4 + 0] = sqfrom; segbuf[nseg * 4 + 1] = sqto; segbuf[nseg * 4 + 2] = hmmfrom; segbuf[nseg * 4 + 3] = hmmto; }
            nseg++;
            in_dom = false;
            __syncwarp();
          }
        }
        if ((s1 == ST_N || s1 == ST_J || s1 == ST_C) && s1 == s0) i--;
        s0 = s1;
      }
      __syncwarp();
      if (failed) continue;
      for (int pos = 1 + lane; pos <= Lr; pos += 32) acc[pos] += val[pos];
      // append this trace's segments left to right
      if (lane == 0) {
        most_in_trace = max(most_in_trace, nseg);
        for (int z = min(nseg, TRCAP) - 1; z >= 0; --z) {
          if (nsp + 0 < SPCAP) {
            int *e = spb + nsp * 5;
            e[0] = t; e[1] = segbuf[z * 4 + 0] + reg.i - 1; e[2] = segbuf[z * 4 + 1] + reg.i - 1; e[3] = segbuf[z * 4 + 2]; e[4] = segbuf[z * 4 + 3];
          }
          nsp++;
        }
        nsp += max(nseg - TRCAP, 0);        // segments the trace buffer had no room for still count towards what is needed
      }
      nsp = __shfl_sync(0xffffffffu, nsp, 0);
      __syncwarp();
    }
    most_in_trace = __shfl_sync(0xffffffffu, most_in_trace, 0);
    const int nsp_all = nsp + 0;
    const bool sp_overflow = nsp > SPCAP || most_in_trace > TRCAP;    // more sampled segments than the buffers hold
    nsp = min(nsp, SPCAP);
    for (int pos = reg.i + lane; pos <= reg.j; pos += 32) n2sc[pos] = (float)log((double)__fdiv_rn(acc[pos - reg.i + 1], (float)NSAMPLES));
    // ---- single-linkage clustering, numbering the clusters exactly as the sequential reference does: seed = last
    // available vertex; pop a vertex, sweep the available list from the top, move every linked vertex to the stack
    // (filling its hole with the list's last element).  The link tests of a sweep run 32 at a time across the lanes;
    // the list surgery is replayed identically by every lane. ----
    int *avail = label, *stack = label + SPCAP, *assign = label + 2 * SPCAP;
    for (int h = lane; h < nsp; h += 32) avail[h] = h;
    __syncwarp();
    int na = nsp, nb = 0, nc = 0;
    while (na > 0) {
      int v = avail[na - 1]; na--;
      stack[nb++] = v;
      while (nb > 0) {
        v = stack[--nb];
        assign[v] = nc;
        for (int base = na - 1; base >= 0; base -= 32) {
          const int pos = base - lane;
          bool linked = false;
          if (pos >= 0) linked = sp_link(spb + v * 5, spb + avail[pos] * 5);
          unsigned mask = __ballot_sync(0xffffffffu, linked);
          while (mask != 0u) {
            const int l = __ffs(mask) - 1;          // lowest lane = highest position first, as the downward sweep does
            mask &= mask - 1;
            const int pz = base - l;
            const int w = avail[pz];
            avail[pz] = avail[na - 1];
            na--;
            stack[nb++] = w;
          }
          __syncwarp();
        }
      }
      nc++;
    }
    __syncwarp();
    // ---- significant clusters -> envelopes (lane 0; the lists are short) ----
    if (lane == 0) {
      int nout = 0;
      Envelope *eo = ep.env_out + ep.env_off[ri];
      for (int c = 0; c < nc; ++c) {
        int idx_of_last = -1, ninc = 0;
        for (int h = 0; h < nsp; ++h) if (assign[h] == c) { if (spb[h * 5] != idx_of_last) ninc++; idx_of_last = spb[h * 5]; }
        if ((float)ninc / (float)NSAMPLES < 0.25f) continue;
        int imin = 1 << 30, jmin = 1 << 30, imax = 0, jmax = 0;
        for (int h = 0; h < nsp; ++h) if (assign[h] == c) {
          imin = min(imin, spb[h * 5 + 1]); imax = max(imax, spb[h * 5 + 1]);
          jmin = min(jmin, spb[h * 5 + 2]); jmax = max(jmax, spb[h * 5 + 2]);
        }
        int cmv, best_i, best_j;
        for (int z = 0; z <= imax - imin; ++z) epc[z] = 0;
        for (int h = 0; h < nsp; ++h) if (assign[h] == c) epc[spb[h * 5 + 1] - imin]++;
        for (cmv = 0, best_i = imin; best_i <= imax; ++best_i) { cmv += epc[best_i - imin]; if ((float)cmv / (float)ninc >= 0.02f) break; }
        for (int z = 0; z <= jmax - jmin; ++z) epc[z] = 0;
        for (int h = 0; h < nsp; ++h) if (assign[h] == c) epc[spb[h * 5 + 2] - jmin]++;
        for (cmv = 0, best_j = jmax; best_j >= jmin; --best_j) { cmv += epc[best_j - jmin]; if ((float)cmv / (float)ninc >= 0.02f) break; }
        if (best_i > best_j) continue;
        if (nout < MAXENV) { eo[nout].pair = reg.pair; eo[nout].i = best_i; eo[nout].j = best_j; eo[nout].null2_done = 1; eo[nout].scratch_off = 0; eo[nout].slot = 0; eo[nout].pad = 0; }
        nout++;                          // counted past MAXENV: the host repeats the region with room for all of them
      }
      const int nsig = nout;
      nout = min(nout, MAXENV);
      // order of occurrence in the target
      for (int a = 1; a < nout; ++a) { Envelope v = eo[a]; int b = a - 1; while (b >= 0 && eo[b].i > v.i) { eo[b + 1] = eo[b]; --b; } eo[b + 1] = v; }
      ep.env_count[ri] = (sp_overflow || nsig > MAXENV) ? -1 : nsig;
      ep.need[ri * 3 + 0] = nsp_all; ep.need[ri * 3 + 1] = most_in_trace; ep.need[ri * 3 + 2] = nsig;
    }
    __syncwarp();
  }
}

// The ensemble of all multi-domain regions as an asynchronous job on stream `st`: ensembles_launch enqueues the uploads,
// the kernel and the downloads; ensembles_collect waits for them and hands back the envelopes of every region.
struct EnsembleJob {
  std::vector<int64_t> off, env_off;
  std::vector<Envelope> envs;
  std::vector<int32_t> cnt, need;
  std::vector<EnsembleCaps> caps;
  int nm = 0;
};

int ensembles_launch(ckm_engine *e, const ckm_models *m, DomdefParams &p, const std::vector<PairWork> &pairs,
                     const std::vector<Region> &regs, const std::vector<int> &multi_idx, const std::vector<EnsembleCaps> &caps,
                     cudaStream_t st, EnsembleJob **job_out) {
  EnsembleJob *job = new EnsembleJob();
  *job_out = job;
  const int nm = job->nm = (int)multi_idx.size();
  job->off.resize(nm); job->env_off.resize(nm); job->caps = caps;
  int64_t tot = 0, nenv = 0;
  for (int i = 0; i < nm; ++i) {
    const Region &r = regs[multi_idx[i]];
    const int64_t Lr = r.j - r.i + 1, M = m->models[pairs[r.pair].model].M, Mpad = ((M + 1) + 31) / 32 * 32 + 32;
    job->off[i] = tot;
    tot += (Lr + 1) * 3 * Mpad + (Lr + 1) * X_NX + 2 * (Lr + 1) + (int64_t)caps[i].segments * 8 + std::max(Lr, M) + 2 + (int64_t)caps[i].trace_segments * 4 + 64;
    tot = (tot + 63) / 64 * 64;
    job->env_off[i] = nenv;
    nenv += caps[i].envelopes;
  }
  // its own keys: the envelope waves run next to it on the class streams
  Region *regs_d; int32_t *idx_d, *cnt_d, *need_d; int64_t *off_d, *eoff_d; float *scr_d; Envelope *env_d; EnsembleCaps *caps_d;
  int rc;
  if ((rc = workspace(e, Ws::EnsRegions, sizeof(Region) * regs.size(), &regs_d)) || (rc = workspace(e, Ws::EnsMultiIdx, sizeof(int32_t) * nm, &idx_d)) ||
      (rc = workspace(e, Ws::EnsScratchOff, sizeof(int64_t) * nm, &off_d)) || (rc = workspace(e, Ws::EnsScratch, sizeof(float) * (size_t)tot, &scr_d)) ||
      (rc = workspace(e, Ws::EnsEnvs, sizeof(Envelope) * (size_t)nenv, &env_d)) || (rc = workspace(e, Ws::EnsCount, sizeof(int32_t) * nm, &cnt_d)) ||
      (rc = workspace(e, Ws::EnsCaps, sizeof(EnsembleCaps) * nm, &caps_d)) || (rc = workspace(e, Ws::EnsEnvOff, sizeof(int64_t) * nm, &eoff_d)) ||
      (rc = workspace(e, Ws::EnsNeed, sizeof(int32_t) * 3 * nm, &need_d))) return rc;
  CKM_CUDA(cudaMemcpyAsync(regs_d, regs.data(), sizeof(Region) * regs.size(), cudaMemcpyHostToDevice, st));       // regs, multi_idx outlive the job (caller)
  CKM_CUDA(cudaMemcpyAsync(idx_d, multi_idx.data(), sizeof(int32_t) * nm, cudaMemcpyHostToDevice, st));
  CKM_CUDA(cudaMemcpyAsync(off_d, job->off.data(), sizeof(int64_t) * nm, cudaMemcpyHostToDevice, st));
  CKM_CUDA(cudaMemcpyAsync(caps_d, job->caps.data(), sizeof(EnsembleCaps) * nm, cudaMemcpyHostToDevice, st));
  CKM_CUDA(cudaMemcpyAsync(eoff_d, job->env_off.data(), sizeof(int64_t) * nm, cudaMemcpyHostToDevice, st));
  CKM_CUDA(cudaMemsetAsync(cnt_d, 0, sizeof(int32_t) * nm, st));
  CKM_CUDA(cudaMemsetAsync(need_d, 0, sizeof(int32_t) * 3 * nm, st));
  CKM_CUDA(cudaMemsetAsync(env_d, 0, sizeof(Envelope) * (size_t)nenv, st));      // the kernel fills only the slots it uses; the whole block is copied back
  EnsembleParams ep;
  ep.d = p; ep.regions = regs_d; ep.multi_idx = idx_d; ep.nmulti = nm;
  ep.scratch_off = off_d; ep.scratch = scr_d; ep.env_out = env_d; ep.env_count = cnt_d;
  ep.caps = caps_d; ep.env_off = eoff_d; ep.need = need_d;
  const size_t smem = (size_t)FWD_WARPS * 3 * p.row_elems * sizeof(float);
  CKM_CUDA(cudaFuncSetAttribute(ensemble_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int grid = std::min(e->prop.multiProcessorCount * 4, (nm + FWD_WARPS - 1) / FWD_WARPS);
  ensemble_kernel<<<grid, FWD_WARPS * 32, smem, st>>>(ep);
  CKM_CUDA(cudaGetLastError());
  e->stats.kernel_launches++;
  job->envs.resize((size_t)nenv);
  job->cnt.resize(nm); job->need.resize((size_t)3 * nm);
  CKM_CUDA(cudaMemcpyAsync(job->envs.data(), env_d, sizeof(Envelope) * job->envs.size(), cudaMemcpyDeviceToHost, st));
  CKM_CUDA(cudaMemcpyAsync(job->cnt.data(), cnt_d, sizeof(int32_t) * nm, cudaMemcpyDeviceToHost, st));
  CKM_CUDA(cudaMemcpyAsync(job->need.data(), need_d, sizeof(int32_t) * 3 * nm, cudaMemcpyDeviceToHost, st));
  return CKM_OK;
}

// out[i]: the envelopes of multi region i.  grow[i]: empty capacities (all zero) when the region fitted, else what it needs:
// the caller repeats the domain phase with them (hmmsearch reports every domain, so must this).
int ensembles_collect(EnsembleJob *job, cudaStream_t st, std::vector<std::vector<Envelope>> &out, std::vector<EnsembleCaps> &grow, int *n_over) {
  cudaError_t err = cudaStreamSynchronize(st);
  *n_over = 0;
  if (err == cudaSuccess) {
    out.assign((size_t)job->nm, {});
    grow.assign((size_t)job->nm, EnsembleCaps{0, 0, 0});
    for (int i = 0; i < job->nm; ++i) {
      if (job->cnt[i] < 0) {
        const EnsembleCaps &c = job->caps[i];
        const bool traces_cut = job->need[3 * i] > c.segments || job->need[3 * i + 1] > c.trace_segments;
        EnsembleCaps g = c;
        g.segments = std::max(c.segments, job->need[3 * i] + 64);
        g.trace_segments = std::max(c.trace_segments, job->need[3 * i + 1] + 8);
        // with the segment list cut short the cluster count is only a lower bound: leave room, the next pass knows exactly
        g.envelopes = std::max(c.envelopes, traces_cut ? std::max(2 * job->need[3 * i + 2], job->need[3 * i + 1] + 8) : job->need[3 * i + 2]);
        grow[i] = g;
        ++*n_over;
        continue;
      }
      for (int c = 0; c < job->cnt[i]; ++c) out[i].push_back(job->envs[(size_t)job->env_off[i] + c]);
    }
  }
  delete job;
  if (err != cudaSuccess) return cuda_fail(err, "ensemble job");
  return CKM_OK;
}
void ensembles_abandon(EnsembleJob *job, cudaStream_t st) { if (job) { cudaStreamSynchronize(st); delete job; } }

}  // namespace ckm
