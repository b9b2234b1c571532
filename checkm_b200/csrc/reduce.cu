// reduce.cu -- the marker-set reduction on the device, for every bin of a finished search:
//   R1  vetHit + addHit                    checkm/resultsParser.py:340-399   (thread per (bin, query) row segment)
//   R2  PFAM clan filter                   checkm/util/pfam.py:86-147        (thread per accepted Pfam hit)
//   R3  list rebuild + adjacent-ORF merge  checkm/resultsParser.py:401-479   (thread per (bin, marker))
//   R4  gene counts, completeness, contamination
//                                          checkm/resultsParser.py:481-537, checkm/markerSets.py:206-238 (thread per bin)
// The reference works on the TEXT of domtblout (checkm/hmmer.py:255-285): scores as "%6.1f", E-values as "%9.2g".
// The kernels apply exactly those roundings to the binary hit records before any comparison, and reproduce the
// reference's list-order semantics (Python dict/list insertion order, stable sort, list.remove) because the
// adjacent-ORF merge depends on them.
#include <algorithm>
#include <cstring>
#include <vector>
#include "engine.hpp"
#include "pool.hpp"

namespace ckm {

struct RRow {                 // one domtblout row as the reference sees it after the text round trip
  int32_t bin, seq, model, tlen, qlen;
  int32_t hmm_from, hmm_to, ali_from, ali_to, env_from, env_to;
  int32_t e_exp, i_exp;       // E-values as mant x 10^(exp-1), mant in 10..99 (0 => E == 0)
  int32_t e_mant, i_mant;
  double  full_score, dom_score;   // rounded to one decimal
};

struct RModel {
  int32_t has_ga, has_tc, has_nc, is_pfam, is_tigr, clan;
  double  ga[2], tc[2], nc[2];
};

struct RParams {
  const ckm_hit *hits; int64_t nhits;
  const double *row_scores;
  RRow *rows;
  const RModel *models;
  const int64_t *nest_off; const int32_t *nest_idx;
  const int32_t *scaffold_id, *orf_num, *name_rank;
  // segments: contiguous rows of one (bin, query)
  const int64_t *seg_off; int32_t nseg;
  const int32_t *seg_bin, *seg_model;
  // R1 outputs
  int32_t *list;              // per row slot: row indices of the accepted hits of the segment, list order
  int32_t *list_len;          // per segment
  // R2 outputs
  uint8_t *filtered;          // per row: dropped by the clan filter
  int64_t *first_app;         // per row: traversal index of the first hit of its ORF (orders rebuilt Pfam lists)
  const int64_t *bin_row_off; // rows of bin b are [bin_row_off[b], bin_row_off[b+1])
  const int64_t *bin_seg_off; // segments of bin b
  // R3 outputs
  ckm_marker_hit *mh; int32_t *mh_len;   // per row slot / per segment
  // R4
  const int64_t *bin_set_off, *set_marker_off; const int32_t *set_marker_idx;
  const int32_t *seg_of_bin_model;       // [nbins][nmodels] -> segment index or -1
  int32_t nbins, nmodels;
  ckm_qa_row *qa;
  ckm_reduce_opts opts;
};

__device__ __forceinline__ void round_evalue(double E, int32_t &ex, int32_t &mant) {
  if (!(E > 0.0)) { ex = INT32_MIN; mant = 0; return; }
  int e = (int)floor(log10(E));
  double m = E / pow(10.0, (double)(e - 1));
  if (m < 10.0) { e -= 1; m = E / pow(10.0, (double)(e - 1)); }
  if (m >= 100.0) { e += 1; m = E / pow(10.0, (double)(e - 1)); }
  double r = rint(m);
  if (r >= 100.0) { r = 10.0; e += 1; }
  ex = e; mant = (int32_t)r;
}

__global__ void r0_round_rows(RParams p) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < p.nhits; i += (int64_t)gridDim.x * blockDim.x) {
    const ckm_hit h = p.hits[i];
    RRow r;
    r.bin = h.bin; r.seq = h.seq; r.model = h.model; r.tlen = h.tlen; r.qlen = h.qlen;
    r.hmm_from = h.hmm_from; r.hmm_to = h.hmm_to; r.ali_from = h.ali_from; r.ali_to = h.ali_to; r.env_from = h.env_from; r.env_to = h.env_to;
    if (p.row_scores != nullptr) { r.full_score = p.row_scores[2 * i]; r.dom_score = p.row_scores[2 * i + 1]; }
    else {
      r.full_score = rint((double)h.full_score * 10.0) / 10.0;
      r.dom_score = rint((double)h.dom_score * 10.0) / 10.0;
    }
    round_evalue(h.full_evalue, r.e_exp, r.e_mant);
    round_evalue(h.i_evalue, r.i_exp, r.i_mant);
    p.rows[i] = r;
    p.filtered[i] = 0;
    p.first_app[i] = -1;
  }
}

__device__ __forceinline__ bool vet_hit(const RParams &p, const RRow &r) {
  const RModel &m = p.models[r.model];
  const ckm_reduce_opts &o = p.opts;
  if (!o.skip_pseudogene) {
    const double alen = (double)(r.ali_to - r.ali_from);
    if (alen / (double)r.qlen < o.pseudogene_length) return false;
  }
  if (m.has_nc && !o.ignore_thresholds && m.is_tigr) return m.nc[0] <= r.full_score && m.nc[1] <= r.dom_score;
  if (m.has_ga && !o.ignore_thresholds) return m.ga[0] <= r.full_score && m.ga[1] <= r.dom_score;
  if (m.has_tc && !o.ignore_thresholds) return m.tc[0] <= r.full_score && m.tc[1] <= r.dom_score;
  if (m.has_nc && !o.ignore_thresholds) return m.nc[0] <= r.full_score && m.nc[1] <= r.dom_score;
  // full_e_value > evalueThreshold, on the 2-significant-digit text value
  bool greater;
  if (r.e_mant == 0) greater = (0.0 > o.evalue_threshold);
  else if (r.e_exp != o.evalue_exp10) greater = r.e_exp > o.evalue_exp10;
  else greater = (double)r.e_mant > o.evalue_mant;
  if (greater) return false;
  const double alen = (double)(r.ali_to - r.ali_from);
  return alen / (double)r.qlen >= o.length_threshold;
}

// R1: one thread per (bin, query) segment walks its rows in file order
__global__ void r1_add_hits(RParams p) {
  for (int s = blockIdx.x * blockDim.x + threadIdx.x; s < p.nseg; s += gridDim.x * blockDim.x) {
    const int64_t r0 = p.seg_off[s], r1 = p.seg_off[s + 1];
    int32_t *lst = p.list + r0;
    int n = 0;
    for (int64_t r = r0; r < r1; ++r) {
      const RRow &row = p.rows[r];
      if (!vet_hit(p, row)) continue;
      int prev = -1;
      for (int z = 0; z < n; ++z) if (p.rows[lst[z]].seq == row.seq) { prev = z; break; }
      if (prev < 0) lst[n++] = (int32_t)r;
      else if (p.rows[lst[prev]].dom_score < row.dom_score) {
        for (int z = prev; z + 1 < n; ++z) lst[z] = lst[z + 1];     // list.remove(previous); list.append(hit)
        lst[n - 1] = (int32_t)r;
      }
    }
    p.list_len[s] = n;
  }
}

__device__ __forceinline__ bool ekey_less(const RRow &a, const RRow &b) {   // (full_e_value, i_evalue) ascending
  if (a.e_exp != b.e_exp) return a.e_exp < b.e_exp;
  if (a.e_mant != b.e_mant) return a.e_mant < b.e_mant;
  if (a.i_exp != b.i_exp) return a.i_exp < b.i_exp;
  return a.i_mant < b.i_mant;
}
__device__ __forceinline__ bool ekey_equal(const RRow &a, const RRow &b) {
  return a.e_exp == b.e_exp && a.e_mant == b.e_mant && a.i_exp == b.i_exp && a.i_mant == b.i_mant;
}

// R2: one thread per accepted Pfam hit rebuilds its ORF's group and replays the clan filter
constexpr int GROUP_CAP = 384;
__global__ void r2_clan_filter(RParams p, int32_t *overflow) {
  for (int s = blockIdx.x * blockDim.x + threadIdx.x; s < p.nseg; s += gridDim.x * blockDim.x) {
    if (!p.models[p.seg_model[s]].is_pfam) continue;
    const int b = p.seg_bin[s];
    const int64_t r0 = p.seg_off[s];
    for (int z = 0; z < p.list_len[s]; ++z) {
      const int32_t me = p.list[r0 + z];
      const int seq = p.rows[me].seq;
      // gather the ORF's Pfam hits in traversal order: segments of the bin in file order, list order inside
      int32_t grp[GROUP_CAP]; int64_t trav[GROUP_CAP]; int g = 0;
      for (int64_t s2 = p.bin_seg_off[b]; s2 < p.bin_seg_off[b + 1]; ++s2) {
        if (!p.models[p.seg_model[s2]].is_pfam) continue;
        const int64_t q0 = p.seg_off[s2];
        for (int y = 0; y < p.list_len[s2]; ++y) {
          const int32_t h = p.list[q0 + y];
          if (p.rows[h].seq != seq) continue;
          if (g < GROUP_CAP) { grp[g] = h; trav[g] = (s2 << 20) + y; }
          g++;
        }
      }
      if (g > GROUP_CAP) { atomicAdd(overflow, 1); g = GROUP_CAP; }
      const int64_t first = trav[0];
      // stable insertion sort by the E-value key
      for (int a = 1; a < g; ++a) {
        const int32_t hv = grp[a]; const int64_t tv = trav[a];
        int c = a - 1;
        while (c >= 0 && ekey_less(p.rows[hv], p.rows[grp[c]])) { grp[c + 1] = grp[c]; trav[c + 1] = trav[c]; --c; }
        grp[c + 1] = hv; trav[c + 1] = tv;
      }
      // replay the filter
      bool dropped[GROUP_CAP];
      for (int a = 0; a < g; ++a) dropped[a] = false;
      for (int a = 0; a < g; ++a) {
        if (dropped[a]) continue;
        const RRow &ri = p.rows[grp[a]];
        const int clanI = p.models[ri.model].clan;
        for (int c = a + 1; c < g; ++c) {
          if (dropped[c]) continue;
          const RRow &rj = p.rows[grp[c]];
          if (clanI != p.models[rj.model].clan) continue;           // two clan-less Pfams (-1 == -1) compare equal
          const bool overlap = (ri.ali_from <= rj.ali_from && ri.ali_to > rj.ali_from) || (rj.ali_from <= ri.ali_from && rj.ali_to > ri.ali_from);
          if (!overlap) continue;
          bool nested = false;
          for (int64_t y = p.nest_off[ri.model]; y < p.nest_off[ri.model + 1]; ++y) if (p.nest_idx[y] == rj.model) { nested = true; break; }
          if (!nested) dropped[c] = true;
        }
      }
      for (int a = 0; a < g; ++a) if (grp[a] == me) { p.filtered[me] = dropped[a] ? 1 : 0; p.first_app[me] = first * 128 + a; }
    }
  }
}

// R3: final list per (bin, marker) and the adjacent-ORF merge
__global__ void r3_adjacent(RParams p) {
  for (int s = blockIdx.x * blockDim.x + threadIdx.x; s < p.nseg; s += gridDim.x * blockDim.x) {
    const int64_t r0 = p.seg_off[s];
    const bool pf = p.models[p.seg_model[s]].is_pfam != 0;
    ckm_marker_hit *mh = p.mh + r0;
    int n = 0;
    // survivors in list order; rebuilt Pfam lists are ordered by their ORF's first appearance (pfam.py:141-145)
    for (int z = 0; z < p.list_len[s]; ++z) {
      const int32_t h = p.list[r0 + z];
      if (pf && p.filtered[h]) continue;
      const RRow &r = p.rows[h];
      ckm_marker_hit v;
      v.bin = r.bin; v.model = r.model; v.seq_a = r.seq; v.seq_b = -1; v.target_length = r.tlen;
      v.hmm_from = r.hmm_from; v.hmm_to = r.hmm_to; v.ali_from = r.ali_from; v.ali_to = r.ali_to; v.env_from = r.env_from; v.env_to = r.env_to;
      v.order = 0; v.src_row = h; v.dict_key = -1;
      int c = n - 1;
      if (pf) { while (c >= 0 && p.first_app[mh[c].src_row] > p.first_app[h]) { mh[c + 1] = mh[c]; --c; } }
      mh[c + 1] = v; n++;
    }
    int64_t dkey = -1;
    if (pf) { dkey = INT64_MAX; for (int z = 0; z < n; ++z) dkey = min(dkey, (int64_t)p.first_app[mh[z].src_row]); }
    if (!p.opts.skip_adjacent) {
      bool combined = true;
      while (combined && n > 0) {
        combined = false;
        for (int i = 0; i < n && !combined; ++i) {
          if (mh[i].seq_b >= 0) continue;                   // a merged name "A&&B" never shares a scaffold id again
          const int scafI = p.scaffold_id[mh[i].seq_a], numI = p.orf_num[mh[i].seq_a];
          int jhit = -1;
          for (int j = i + 1; j < n; ++j) {
            if (mh[j].seq_b >= 0) continue;
            if (p.scaffold_id[mh[j].seq_a] != scafI) continue;
            const int numJ = p.orf_num[mh[j].seq_a];
            if (numI == INT32_MIN || numJ == INT32_MIN) break;      // int() raised: leave the j loop
            const long long d = (long long)numI - (long long)numJ;
            if (d == 1 || d == -1) { jhit = j; break; }
          }
          if (jhit >= 0) {
            ckm_marker_hit nh = mh[i];
            const ckm_marker_hit &hj = mh[jhit];
            const bool a_first = p.name_rank[nh.seq_a] <= p.name_rank[hj.seq_a];
            const int sa = a_first ? nh.seq_a : hj.seq_a, sb = a_first ? hj.seq_a : nh.seq_a;
            nh.seq_a = sa; nh.seq_b = sb;
            nh.target_length = mh[i].target_length + hj.target_length;
            nh.hmm_from = min(mh[i].hmm_from, hj.hmm_from); nh.hmm_to = min(mh[i].hmm_to, hj.hmm_to);
            nh.ali_from = min(mh[i].ali_from, hj.ali_from); nh.ali_to = min(mh[i].ali_to, hj.ali_to);
            nh.env_from = min(mh[i].env_from, hj.env_from); nh.env_to = min(mh[i].env_to, hj.env_to);
            // hits.remove(hits[j]); hits.remove(hits[i]); hits.append(newHit)
            int w = 0;
            for (int z = 0; z < n; ++z) if (z != i && z != jhit) mh[w++] = mh[z];
            mh[w++] = nh;
            n = w;
            combined = true;
          }
        }
      }
    }
    for (int z = 0; z < n; ++z) { mh[z].order = z; mh[z].dict_key = dkey; }
    p.mh_len[s] = n;
  }
}

// R4: gene counts + completeness/contamination per bin
__global__ void r4_counts(RParams p) {
  for (int b = blockIdx.x * blockDim.x + threadIdx.x; b < p.nbins; b += gridDim.x * blockDim.x) {
    ckm_qa_row q;
    q.bin = b;
    for (int z = 0; z < 6; ++z) q.counts[z] = 0;
    q.n_markers = 0; q.n_sets = (int32_t)(p.bin_set_off[b + 1] - p.bin_set_off[b]);
    q.unique_hits = 0; q.multi_hits = 0;
    // countUniqueHits runs over every marker that has hits, in or out of the selected set
    for (int64_t s = p.bin_seg_off[b]; s < p.bin_seg_off[b + 1]; ++s) {
      const int n = p.mh_len[s];
      if (n == 1) q.unique_hits++; else if (n > 1) q.multi_hits++;
    }
    double comp = 0.0, cont = 0.0;
    int present_all = 0, multi_all = 0;
    for (int64_t st = p.bin_set_off[b]; st < p.bin_set_off[b + 1]; ++st) {
      int present = 0, multi = 0;
      const int64_t m0 = p.set_marker_off[st], m1 = p.set_marker_off[st + 1];
      for (int64_t y = m0; y < m1; ++y) {
        const int model = p.set_marker_idx[y];
        const int seg = (model >= 0) ? p.seg_of_bin_model[(int64_t)b * p.nmodels + model] : -1;
        const int cnt = (seg >= 0) ? p.mh_len[seg] : 0;
        q.counts[min(cnt, 5)]++;
        q.n_markers++;
        if (cnt >= 1) { present++; multi += cnt - 1; }
      }
      present_all += present; multi_all += multi;
      comp += (double)present / (double)(m1 - m0);
      cont += (double)multi / (double)(m1 - m0);
    }
    if (p.opts.individual_markers) {
      q.completeness = 100.0 * (double)present_all / (double)q.n_markers;
      q.contamination = 100.0 * (double)multi_all / (double)q.n_markers;
    } else {
      q.completeness = 100.0 * comp / (double)q.n_sets;
      q.contamination = 100.0 * cont / (double)q.n_sets;
    }
    p.qa[b] = q;
  }
}

// genomeCheck on explicit copy numbers (thread per bin)
__global__ void genome_check_kernel(int32_t nbins, const int64_t *bin_set_off, const int64_t *set_marker_off, const int32_t *cnts,
                                    int32_t individual, ckm_qa_row *out) {
  for (int b = blockIdx.x * blockDim.x + threadIdx.x; b < nbins; b += gridDim.x * blockDim.x) {
    ckm_qa_row q;
    q.bin = b;
    for (int z = 0; z < 6; ++z) q.counts[z] = 0;
    q.n_markers = 0; q.n_sets = (int32_t)(bin_set_off[b + 1] - bin_set_off[b]); q.unique_hits = 0; q.multi_hits = 0;
    double comp = 0.0, cont = 0.0; int present_all = 0, multi_all = 0;
    for (int64_t st = bin_set_off[b]; st < bin_set_off[b + 1]; ++st) {
      int present = 0, multi = 0;
      const int64_t m0 = set_marker_off[st], m1 = set_marker_off[st + 1];
      for (int64_t y = m0; y < m1; ++y) {
        const int cnt = cnts[y];
        q.counts[min(cnt, 5)]++; q.n_markers++;
        if (cnt == 1) q.unique_hits++; else if (cnt > 1) q.multi_hits++;
        if (cnt >= 1) { present++; multi += cnt - 1; }
      }
      present_all += present; multi_all += multi;
      comp += (double)present / (double)(m1 - m0);
      cont += (double)multi / (double)(m1 - m0);
    }
    if (individual) { q.completeness = 100.0 * (double)present_all / (double)q.n_markers; q.contamination = 100.0 * (double)multi_all / (double)q.n_markers; }
    else { q.completeness = 100.0 * comp / (double)q.n_sets; q.contamination = 100.0 * cont / (double)q.n_sets; }
    out[b] = q;
  }
}

// Device buffers of one call, from the stream-ordered pool (none of them stays resident), handed back to it stream-ordered (no
// device-wide synchronisation) when the holder goes out of scope.
struct CallBuffers {
  cudaStream_t st; const char *who;
  std::vector<void *> held;
  CallBuffers(cudaStream_t s, const char *w) : st(s), who(w) {}
  CallBuffers(const CallBuffers &) = delete;
  ~CallBuffers() { for (void *q : held) cudaFreeAsync(q, st); }
  // n elements (at least 16 bytes); CKM_ENOMEM when the device has no room.  upload: filled from the host.
  template <class T> int get(T **out, size_t n) {
    void *q = nullptr;
    if (cudaMallocAsync(&q, std::max<size_t>(sizeof(T) * n, 16), st) != cudaSuccess) { set_error(std::string(who) + ": out of device memory"); return CKM_ENOMEM; }
    held.push_back(q); *out = static_cast<T *>(q);
    return CKM_OK;
  }
  template <class T> int upload(T **out, const void *src, size_t n) {
    const int rc = get(out, n);
    if (rc == CKM_OK && n > 0) CKM_CUDA(cudaMemcpyAsync((void *)*out, src, sizeof(T) * n, cudaMemcpyHostToDevice, st));
    return rc;
  }
};

}  // namespace ckm

using namespace ckm;

extern "C" int ckm_genome_check(ckm_engine *e, int32_t nbins, const int64_t *bin_set_off, const int64_t *set_marker_off,
                                const int32_t *marker_count, int32_t individual_markers, ckm_qa_row *rows_out) {
  if (!e || nbins < 0 || !bin_set_off || !set_marker_off || !rows_out) { set_error("ckm_genome_check: bad argument"); return CKM_EINVAL; }
  if (nbins == 0) return CKM_OK;
  cudaSetDevice(e->device);
  cudaStream_t st = e->stream;
  const int64_t nsets = bin_set_off[nbins], nm = set_marker_off[nsets];
  CallBuffers mem(st, "ckm_genome_check");
  int64_t *d_b, *d_s; int32_t *d_c; ckm_qa_row *d_o;
  int rc;
  if ((rc = mem.upload(&d_b, bin_set_off, (size_t)nbins + 1)) || (rc = mem.upload(&d_s, set_marker_off, (size_t)(nsets + 1))) ||
      (rc = mem.upload(&d_c, marker_count, (size_t)nm)) || (rc = mem.get(&d_o, (size_t)nbins))) return rc;
  genome_check_kernel<<<(nbins + 127) / 128, 128, 0, st>>>(nbins, d_b, d_s, d_c, individual_markers, d_o);
  CKM_CUDA(cudaGetLastError());
  CKM_CUDA(cudaMemcpyAsync(rows_out, d_o, sizeof(ckm_qa_row) * nbins, cudaMemcpyDeviceToHost, st));
  CKM_CUDA(cudaStreamSynchronize(st));
  e->stats.kernel_launches++;
  return CKM_OK;
}


static int reduce_once(ckm_engine *e, int32_t nmodels_in, int32_t nseq_in, int32_t nbins_in, const ckm_hit *hits, int64_t nhits,
                       const ckm_reduce_opts *opts, const ckm_reduce_meta *meta,
                       ckm_qa_row **qa_out, int32_t *nqa_out, ckm_marker_hit **mh_out, int64_t *nmh_out) {
  if (!e || nmodels_in < 0 || nseq_in < 0 || nbins_in < 1 || !opts || !meta || !qa_out || !nqa_out || !mh_out || !nmh_out || (nhits > 0 && !hits)) { set_error("ckm_reduce: bad argument"); return CKM_EINVAL; }
  cudaSetDevice(e->device);
  cudaStream_t st = e->stream;
  const int nbins = nbins_in, nmodels = nmodels_in, nseq = nseq_in;
  *qa_out = nullptr; *mh_out = nullptr; *nqa_out = 0; *nmh_out = 0;
  // segments = maximal runs of equal (bin, model); rows of a bin must be contiguous and bins ascending (ckm_search order)
  std::vector<int64_t> seg_off{0}, bin_row_off(nbins + 1, 0), bin_seg_off(nbins + 1, 0);
  std::vector<int32_t> seg_bin, seg_model, seg_of((size_t)nbins * nmodels, -1);
  for (int64_t i = 0; i < nhits; ++i) {
    if (hits[i].bin < 0 || hits[i].bin >= nbins || hits[i].model < 0 || hits[i].model >= nmodels || hits[i].seq < 0 || hits[i].seq >= nseq) { set_error("ckm_reduce: hit row out of range"); return CKM_EINVAL; }
    if (i > 0 && hits[i].bin < hits[i - 1].bin) { set_error("ckm_reduce: hit rows must be grouped by bin in ascending order"); return CKM_EINVAL; }
    if (i == 0 || hits[i].bin != hits[i - 1].bin || hits[i].model != hits[i - 1].model) {
      if (i > 0) seg_off.push_back(i);
      seg_bin.push_back(hits[i].bin); seg_model.push_back(hits[i].model);
      int32_t &slot = seg_of[(size_t)hits[i].bin * nmodels + hits[i].model];
      if (slot >= 0) { set_error("ckm_reduce: rows of one (bin, query) must be contiguous"); return CKM_EINVAL; }
      slot = (int32_t)seg_bin.size() - 1;
    }
    bin_row_off[hits[i].bin + 1] = i + 1;
  }
  if (nhits > 0) seg_off.push_back(nhits);
  const int nseg = (int)seg_bin.size();
  for (int b = 0; b < nbins; ++b) if (bin_row_off[b + 1] < bin_row_off[b]) bin_row_off[b + 1] = bin_row_off[b];
  { int s = 0; for (int b = 0; b < nbins; ++b) { bin_seg_off[b] = s; while (s < nseg && seg_bin[s] == b) ++s; } bin_seg_off[nbins] = s; }
  std::vector<RModel> rm(nmodels);
  for (int i = 0; i < nmodels; ++i) {
    RModel &r = rm[i];
    r.has_ga = meta->has_cut ? meta->has_cut[i * 3 + 0] : 0; r.has_tc = meta->has_cut ? meta->has_cut[i * 3 + 1] : 0; r.has_nc = meta->has_cut ? meta->has_cut[i * 3 + 2] : 0;
    r.is_pfam = meta->is_pfam ? meta->is_pfam[i] : 0; r.is_tigr = meta->is_tigr ? meta->is_tigr[i] : 0; r.clan = meta->clan ? meta->clan[i] : -1;
    for (int z = 0; z < 2; ++z) { r.ga[z] = meta->cutoffs ? meta->cutoffs[i * 6 + z] : 0.0; r.tc[z] = meta->cutoffs ? meta->cutoffs[i * 6 + 2 + z] : 0.0; r.nc[z] = meta->cutoffs ? meta->cutoffs[i * 6 + 4 + z] : 0.0; }
  }
  std::vector<int64_t> nest_off_default(nmodels + 1, 0);
  const int64_t *nest_off = meta->nest_off ? meta->nest_off : nest_off_default.data();
  const int64_t nnest = nest_off[nmodels];
  const int64_t nsets = meta->bin_set_off ? meta->bin_set_off[nbins] : 0;
  const int64_t nsetm = (meta->set_marker_off && nsets > 0) ? meta->set_marker_off[nsets] : 0;
  std::vector<int64_t> zero_off(nbins + 1, 0), zero_set(1, 0);

  RParams p;
  std::memset(&p, 0, sizeof(p));
  p.nhits = nhits; p.nseg = nseg; p.nbins = nbins; p.nmodels = nmodels; p.opts = *opts;
  const size_t nh = (size_t)std::max<int64_t>(nhits, 1), ns = (size_t)std::max(nseg, 1);
  CallBuffers mem(st, "ckm_reduce");
  int32_t *d_overflow;
  int rc;
  if ((rc = mem.upload(&p.hits, hits, (size_t)nhits))) return rc;
  if (meta->row_scores != nullptr && nhits > 0 && (rc = mem.upload(&p.row_scores, meta->row_scores, 2 * (size_t)nhits))) return rc;
  if ((rc = mem.get(&p.rows, nh)) || (rc = mem.get(&p.list, nh)) || (rc = mem.get(&p.list_len, ns)) || (rc = mem.get(&p.filtered, nh)) ||
      (rc = mem.get(&p.first_app, nh)) || (rc = mem.get(&p.mh, nh)) || (rc = mem.get(&p.mh_len, ns)) || (rc = mem.get(&p.qa, (size_t)nbins)) ||
      (rc = mem.get(&d_overflow, 1))) return rc;
  CKM_CUDA(cudaMemsetAsync(d_overflow, 0, sizeof(int32_t), st));
  CKM_CUDA(cudaMemsetAsync(p.mh_len, 0, sizeof(int32_t) * ns, st));
  std::vector<int32_t> zero_seq(std::max(nseq, 1), 0);
  if ((rc = mem.upload(&p.models, rm.data(), rm.size())) || (rc = mem.upload(&p.nest_off, nest_off, (size_t)nmodels + 1)) ||
      (rc = mem.upload(&p.nest_idx, meta->nest_idx, (size_t)nnest)) ||
      (rc = mem.upload(&p.scaffold_id, meta->scaffold_id ? meta->scaffold_id : zero_seq.data(), (size_t)nseq)) ||
      (rc = mem.upload(&p.orf_num, meta->orf_num ? meta->orf_num : zero_seq.data(), (size_t)nseq)) ||
      (rc = mem.upload(&p.name_rank, meta->name_rank ? meta->name_rank : zero_seq.data(), (size_t)nseq)) ||
      (rc = mem.upload(&p.seg_off, seg_off.data(), seg_off.size())) || (rc = mem.upload(&p.seg_bin, seg_bin.data(), seg_bin.size())) ||
      (rc = mem.upload(&p.seg_model, seg_model.data(), seg_model.size())) || (rc = mem.upload(&p.bin_row_off, bin_row_off.data(), bin_row_off.size())) ||
      (rc = mem.upload(&p.bin_seg_off, bin_seg_off.data(), bin_seg_off.size())) ||
      (rc = mem.upload(&p.bin_set_off, meta->bin_set_off ? meta->bin_set_off : zero_off.data(), (size_t)nbins + 1)) ||
      (rc = mem.upload(&p.set_marker_off, (meta->set_marker_off && nsets > 0) ? meta->set_marker_off : zero_set.data(), (size_t)(nsets + 1))) ||
      (rc = mem.upload(&p.set_marker_idx, meta->set_marker_idx, (size_t)nsetm)) ||
      (rc = mem.upload(&p.seg_of_bin_model, seg_of.data(), seg_of.size()))) return rc;

  const int T = 128;
  if (nhits > 0) {
    r0_round_rows<<<(int)std::min<int64_t>((nhits + T - 1) / T, 4096), T, 0, st>>>(p);
    r1_add_hits<<<(nseg + T - 1) / T, T, 0, st>>>(p);
    r2_clan_filter<<<(nseg + 31) / 32, 32, 0, st>>>(p, d_overflow);
    r3_adjacent<<<(nseg + T - 1) / T, T, 0, st>>>(p);
  }
  r4_counts<<<(nbins + T - 1) / T, T, 0, st>>>(p);
  CKM_CUDA(cudaGetLastError());
  e->stats.kernel_launches += 5;
  std::vector<ckm_marker_hit> mh((size_t)nhits);
  std::vector<int32_t> mh_len(std::max(nseg, 1), 0);
  ckm_qa_row *qa = (ckm_qa_row *)std::malloc(sizeof(ckm_qa_row) * std::max(nbins, 1));
  int32_t overflow = 0;
  if (nhits > 0) {
    CKM_CUDA(cudaMemcpyAsync(mh.data(), p.mh, sizeof(ckm_marker_hit) * (size_t)nhits, cudaMemcpyDeviceToHost, st));
    CKM_CUDA(cudaMemcpyAsync(mh_len.data(), p.mh_len, sizeof(int32_t) * nseg, cudaMemcpyDeviceToHost, st));
  }
  CKM_CUDA(cudaMemcpyAsync(qa, p.qa, sizeof(ckm_qa_row) * nbins, cudaMemcpyDeviceToHost, st));
  CKM_CUDA(cudaMemcpyAsync(&overflow, d_overflow, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  CKM_CUDA(cudaStreamSynchronize(st));
  if (overflow) { std::free(qa); set_error("ckm_reduce: more than 384 Pfam hits on one ORF"); return CKM_ECAPACITY; }
  // compact the per-segment lists
  int64_t total = 0;
  for (int s = 0; s < nseg; ++s) total += mh_len[s];
  ckm_marker_hit *out = (ckm_marker_hit *)std::malloc(sizeof(ckm_marker_hit) * (size_t)std::max<int64_t>(total, 1));
  int64_t w = 0;
  for (int s = 0; s < nseg; ++s)
    for (int z = 0; z < mh_len[s]; ++z) out[w++] = mh[(size_t)seg_off[s] + z];
  *qa_out = qa; *nqa_out = nbins; *mh_out = out; *nmh_out = total;
  return CKM_OK;
}

// Frees what the engine keeps cached between calls: its workspaces (the next call allocates them again) and the unused blocks
// of the device's stream-ordered pool.
static void release_cached_memory(ckm_engine *e) {
  cudaStreamSynchronize(e->stream);
  for (auto &s : e->cls) cudaStreamSynchronize(s);
  if (e->aux) cudaStreamSynchronize(e->aux);
  workspace_release(e);
  cudaMemPool_t mp;
  if (cudaDeviceGetDefaultMemPool(&mp, e->device) == cudaSuccess) cudaMemPoolTrimTo(mp, 0);
}

extern "C" int ckm_reduce(ckm_engine *e, int32_t nmodels_in, int32_t nseq_in, int32_t nbins_in, const ckm_hit *hits, int64_t nhits,
                          const ckm_reduce_opts *opts, const ckm_reduce_meta *meta,
                          ckm_qa_row **qa_out, int32_t *nqa_out, ckm_marker_hit **mh_out, int64_t *nmh_out) {
  int rc = reduce_once(e, nmodels_in, nseq_in, nbins_in, hits, nhits, opts, meta, qa_out, nqa_out, mh_out, nmh_out);
  if (rc == CKM_ENOMEM) {
    // after a large search the engine's workspaces can hold most of the device: a reduction over many bins
    // (one analyseResults over a whole directory) then finds no room for its rows
    cudaGetLastError();              // the failed allocation must not surface as a launch error of the retry
    release_cached_memory(e);
    rc = reduce_once(e, nmodels_in, nseq_in, nbins_in, hits, nhits, opts, meta, qa_out, nqa_out, mh_out, nmh_out);
  }
  return rc;
}
