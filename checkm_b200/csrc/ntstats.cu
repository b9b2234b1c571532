// ntstats.cu -- base composition and contig structure of a bin's scaffolds: the integer half of CheckM's bin statistics
// (checkm/binStatistics.py:176-243: calculateGC, calculateSeqStats; SURVEY.md 8 row f4).  Everything here is a byte scan
// bound by HBM: 2 KB rows stream through shared memory by TMA bulk copies, one warp per row, a lane takes 64 consecutive bytes.
//
// What the reference computes per scaffold, restated as local predicates:
//   * a, c, g, t: case-insensitive counts, U counted with T (util/seqUtils.py:279-286)
//   * ambiguous bases: count('N') + count('n')
//   * contigs: scaffold.split('N' * 10), the remaining 'N' of every piece deleted, empty pieces dropped.  A maximal run of
//     r upper-case N holds floor(r / 10) separators and the other N are deleted anyway, so the pieces are exactly the
//     stretches between runs of >= 10 N, and a piece's length is its number of bytes that are not 'N'.
//     Position i ends such a run iff bytes i-9..i are all 'N' and byte i+1 is not (or the scaffold ends): a predicate with a
//     9-byte halo.  The contig index of a byte is the number of run ends before it (a prefix sum), the contig length a
//     histogram over that index.
#include <cstdint>
#include <cstring>
#include <numeric>
#include <vector>
#include "engine.hpp"
#include "pool.hpp"
#include "device_utils.cuh"

using namespace ckm;

namespace {

constexpr int NT_THREADS = 256;
constexpr int NT_WARPS = NT_THREADS / 32;
constexpr int NT_CHUNK = 64;                         // bytes of one lane in one row: one bit each in a 64-bit mask
constexpr int NT_ROW = 32 * NT_CHUNK;                // 2 KB: what a warp takes at a time
constexpr int NT_HALO = 16;                          // bytes staged either side of a row (9 before and 1 after are looked at)
constexpr int NT_STAGE = NT_HALO + NT_ROW + NT_HALO;
constexpr int NT_STAGES = 3;                         // rows in flight per warp
constexpr int NT_DESC_OFF = NT_STAGES * NT_STAGE;    // per-warp shared memory: the stages, their row descriptors, their mbarriers
constexpr int NT_BAR_OFF = NT_DESC_OFF + NT_STAGES * 16;
constexpr int NT_WARP_SMEM = (NT_BAR_OFF + NT_STAGES * 8 + 127) / 128 * 128;
#ifndef CKM_NT_CTAS
#define CKM_NT_CTAS 4
#endif
constexpr int NT_CTAS_PER_SM = CKM_NT_CTAS;          // 4: 32 warps x 3 x 2 KB of stages = 200 KB of shared memory, <= 64 registers

// The scaffolds of a call, cut into 2 KB rows, form one list; every warp of the grid takes a contiguous range of it and
// streams its rows through its own ring of shared-memory stages, filled by TMA bulk copies that lane 0 issues NT_STAGES
// ahead.  Warps never wait for each other.  A "piece" is the part of one scaffold inside one warp's range.  Contigs closed
// inside a piece are reported by the kernel; the bases before the first run end of a piece (head) and after its last (tail)
// come back separately and the host joins tail + head across the cuts (ckm_scaffold_stats below).
// Piece index = scaffold + warp: along the list one of the two grows at every cut.
// src: device address the row's copy starts at (16 bytes before the row unless it is the first of its scaffold);
// info: valid bytes (1..2048) | 16-byte units of the copy << 12 | first row << 30 | last row << 31
struct NtRow { uint64_t src; uint32_t scaf; uint32_t info; };
struct NtPiece { uint32_t head, tail, closed, pad; };              // closed: the piece holds at least one run end

struct NtParams {
  const uint8_t *bytes;            // every scaffold starts at a multiple of 64 and is followed by padding up to the next one
  const NtRow *rows;
  long long nrows;
  NtPiece *piece;                  // nscaf + warps of the grid, zeroed
  unsigned long long *stats;       // nscaf x 8: a c g t N n contigs contig_bases (the last two: contigs closed inside pieces)
  uint32_t *contig_scaf, *contig_len;
  unsigned long long *ncontigs;
  long long cap;
};

// 0x80 in every byte of w that equals the byte replicated in pat
__device__ __forceinline__ uint32_t eq4(uint32_t w, uint32_t pat) {
  const uint32_t x = w ^ pat;
  const uint32_t t = (x & 0x7F7F7F7Fu) + 0x7F7F7F7Fu;
  return ~(t | x | 0x7F7F7F7Fu);
}
// the four 0x80 flags of eq4 as a 4-bit mask, byte 0 -> bit 0
__device__ __forceinline__ uint32_t nibble(uint32_t flags) { return (((flags >> 7) * 0x01020408u) >> 24) & 0xFu; }
// sum of the four bytes of x (the sum must stay below 256)
__device__ __forceinline__ uint32_t hsum4(uint32_t x) { return (x * 0x01010101u) >> 24; }

// lane 0: hand a stage to the copy engine.  Every value loaded from the stage has been used by now, so the loads are done.
__device__ __forceinline__ void nt_issue(const NtRow d, uint32_t stage, uint32_t desc, uint32_t bar) {
  asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(desc), "r"((uint32_t)d.src), "r"((uint32_t)(d.src >> 32)), "r"(d.scaf), "r"(d.info) : "memory");
  const uint32_t bytes = ((d.info >> 12) & 0xFFu) * 16u;
  fence_proxy_async();
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(stage + (((d.info >> 30) & 1u) ? (uint32_t)NT_HALO : 0u)),
               "l"(d.src), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ void nt_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "NT_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra NT_DONE;\n"
      "bra NT_WAIT;\n"
      "NT_DONE:\n"
      "}\n" ::"r"(bar), "r"(parity) : "memory");
}

__device__ __forceinline__ void nt_emit(const NtParams &p, uint32_t scaf, uint32_t len) {
  if (len == 0) return;
  const unsigned long long at = atomicAdd(p.ncontigs, 1ull);
  if ((long long)at < p.cap) { p.contig_scaf[at] = scaf; p.contig_len[at] = len; }
  atomicAdd(&p.stats[(size_t)scaf * 8 + 6], 1ull);
  atomicAdd(&p.stats[(size_t)scaf * 8 + 7], (unsigned long long)len);
}

__global__ void __launch_bounds__(NT_THREADS, NT_CTAS_PER_SM) ntstats_kernel(NtParams p) {
  extern __shared__ __align__(128) uint8_t s_dyn[];             // NT_WARPS x NT_WARP_SMEM
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long long gw = (long long)blockIdx.x * NT_WARPS + warp, nw = (long long)gridDim.x * NT_WARPS;
  const long long lo = p.nrows * gw / nw, hi = p.nrows * (gw + 1) / nw;
  if (lo >= hi) return;
  const int n = (int)(hi - lo);                                  // rows of this warp (the host keeps a call below 2^31 rows)
  const NtRow *mine = p.rows + lo;
  const uint32_t ring = smem_u32(s_dyn) + warp * NT_WARP_SMEM;     // stage i at ring + i * NT_STAGE
  NtRow upcoming = {0, 0u, 0u};                                  // lane 0: the row to issue next, fetched one row early
  if (lane == 0) {
    for (int i = 0; i < NT_STAGES; ++i) asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(ring + NT_BAR_OFF + i * 8) : "memory");
    fence_mbar_init();
    for (int i = 0; i < NT_STAGES && i < n; ++i) nt_issue(mine[i], ring + i * NT_STAGE, ring + NT_DESC_OFF + i * 16, ring + NT_BAR_OFF + i * 8);
    if (NT_STAGES < n) upcoming = mine[NT_STAGES];
  }
  __syncwarp();
  const int rot = (lane >> 1) & 3;                               // the lane reads its four 16-byte vectors starting at this one:
                                                                 // eight neighbouring lanes then touch eight different bank groups
  uint32_t cA = 0, cC = 0, cG = 0, cT = 0, cN = 0, cn = 0;       // per-lane counts over the piece
  uint32_t carry = 0;                                            // bases of the contig still open (same in every lane)
  uint32_t head = 0; bool closed = false;                        // same in every lane
  int st = 0; uint32_t phase = 0;
  uint32_t tail9 = 0;                                            // lane 0: is-N of the nine bytes before the row
  for (int k = 0; k < n; ++k) {
    nt_wait(ring + NT_BAR_OFF + st * 8, phase);
    const uint4 d = lds128(ring + NT_DESC_OFF + st * 16);
    const uint32_t s = d.z;
    const int nbytes = (int)(d.w & 0xFFFu);
    const bool first_row = (d.w >> 30) & 1u, last_row = (d.w >> 31) != 0;
    const uint32_t body = ring + st * NT_STAGE + NT_HALO;
    const int left = nbytes - lane * NT_CHUNK;                   // bytes of the scaffold in and after this lane's chunk
    uint32_t w[16];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const uint4 v = lds128(body + lane * NT_CHUNK + ((q + rot) & 3) * 16);
      w[4 * q] = v.x; w[4 * q + 1] = v.y; w[4 * q + 2] = v.z; w[4 * q + 3] = v.w;
    }
    // halo, read before the stage is handed back: is-N of the byte after the row, and -- only at the first row of this warp's
    // range, afterwards the previous row's mask is at hand -- of the 12 bytes before it
    uint32_t halo_bits = 0;
    if (k == 0 && lane == 0 && !first_row) {
      const uint4 v = lds128(body - NT_HALO);
      halo_bits = nibble(eq4(v.y, 0x4E4E4E4Eu)) | (nibble(eq4(v.z, 0x4E4E4E4Eu)) << 4) | (nibble(eq4(v.w, 0x4E4E4E4Eu)) << 8);
      tail9 = halo_bits >> 3;                                    // bytes -12..-1 -> the last nine
    }
    if (lane == 31 && !last_row) halo_bits = s_dyn[warp * NT_WARP_SMEM + st * NT_STAGE + NT_HALO + NT_ROW] == 'N';

    unsigned long long m = 0, valid = 0;
    if (left > 0) {
      valid = left >= NT_CHUNK ? ~0ull : ((1ull << left) - 1ull);
      if (left < NT_CHUNK) {                    // last chunk of the scaffold: whatever the padding holds is not sequence;
#pragma unroll                                  // count it as 'A' here and take it off again below
        for (int j = 0; j < 16; ++j) {
          const int keep = left - ((((j >> 2) + rot) & 3) * 16 + (j & 3) * 4);   // bytes of this word inside the scaffold
          if (keep < 4) { const uint32_t in = keep <= 0 ? 0u : ((1u << (8 * keep)) - 1u); w[j] = (w[j] & in) | (0x41414141u & ~in); }
        }
      }
      // Fast path, a chunk of nothing but upper-case A C G T (what assemblies mostly are): the low three bits of the
      // four letters differ (A 1, C 3, T 4, G 7), so one byte permute looks up the letter each byte would have to be and
      // one xor tells whether it is.  Two more permutes by the same index look up what the byte adds to the counts:
      // 0x01 for C, 0x10 for G in one table (two 4-bit counters per byte lane, 8 words each), 0x01 for T in the other.
      uint32_t bad = 0, cg0 = 0, cg1 = 0, tt = 0;
#pragma unroll
      for (int j = 0; j < 16; ++j) {
        uint32_t t = w[j] & 0x07070707u;
        t |= t >> 4;
        const uint32_t sel = prmt_b32(t, 0u, 0x4420);           // the four 3-bit indices as selector nibbles (all below 8)
        bad |= w[j] ^ prmt_b32(0x43FF41FFu, 0x47FFFF54u, sel);
        const uint32_t cg = prmt_b32(0x01000000u, 0x10000000u, sel);
        if (j < 8) cg0 += cg; else cg1 += cg;
        tt += prmt_b32(0u, 0x00000001u, sel);
      }
      if (bad == 0) {
        const uint32_t nc = hsum4((cg0 & 0x0F0F0F0Fu) + (cg1 & 0x0F0F0F0Fu)), ng = hsum4(((cg0 >> 4) & 0x0F0F0F0Fu) + ((cg1 >> 4) & 0x0F0F0F0Fu));
        const uint32_t nt = hsum4(tt);
        cC += nc; cG += ng; cT += nt; cA += (uint32_t)min(left, NT_CHUNK) - nc - ng - nt;
      } else {
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          const int first = (((j >> 2) + rot) & 3) * 16 + (j & 3) * 4;      // where the word sits in the chunk
          uint32_t x = w[j];
          if (left < first + 4) {               // the padding stand-ins again
            const int keep = left - first;
            x = keep <= 0 ? 0u : (x & ((1u << (8 * keep)) - 1u));
          }
          const uint32_t up = x & 0xDFDFDFDFu;             // 'a' -> 'A'; no other byte maps onto a letter tested below
          cA += __popc(eq4(up, 0x41414141u));
          cC += __popc(eq4(up, 0x43434343u));
          cG += __popc(eq4(up, 0x47474747u));
          cT += __popc(eq4(up, 0x54545454u)) + __popc(eq4(up, 0x55555555u));
          const uint32_t fN = eq4(x, 0x4E4E4E4Eu);
          cN += __popc(fN);
          cn += __popc(eq4(x, 0x6E6E6E6Eu));
          m |= (unsigned long long)nibble(fN) << first;
        }
      }
    }
    // halo: is-N of the 9 bytes before this chunk and of the byte after it
    const uint32_t up9 = __shfl_up_sync(0xffffffffu, (uint32_t)(m >> 55), 1);
    const uint32_t dn1 = __shfl_down_sync(0xffffffffu, (uint32_t)(m & 1ull), 1);
    const uint32_t after = __shfl_sync(0xffffffffu, halo_bits, 31);           // (also: the halo byte has been loaded and used)
    const unsigned long long prev9 = lane > 0 ? up9 : (first_row ? 0u : tail9);
    const unsigned long long nextbit = lane < 31 ? dn1 : after;
    if (!__any_sync(0xffffffffu, (m | prev9) != 0ull)) {
      carry += (uint32_t)nbytes;                                 // not an N in sight: the whole row belongs to the open contig
    } else {
      unsigned long long ends = 0;
      if (m | prev9) {
        const unsigned __int128 X = ((unsigned __int128)m << 9) | (unsigned __int128)prev9;
        const unsigned __int128 A = X & (X >> 1), B = A & (A >> 2), C8 = B & (B >> 4);
        const unsigned long long run10 = (unsigned long long)(C8 & (A >> 8));   // bit i: bytes i-9 .. i of the chunk are all N
        ends = run10 & ~((m >> 1) | (nextbit << 63)) & valid;
      }
      const unsigned long long bases = valid & ~m;
      // per lane: bases up to its first run end (all of them if it has none), bases after its last; contigs between two run
      // ends of the same lane are complete and reported here
      const bool has = ends != 0ull;
      uint32_t pre = __popcll(bases), post = 0;
      if (has) {
        unsigned long long rest = bases, e = ends;
        int b = __ffsll((long long)e) - 1;
        unsigned long long upto = b == 63 ? ~0ull : ((2ull << b) - 1ull);
        pre = __popcll(rest & upto); rest &= ~upto; e &= e - 1;
        while (e) {
          b = __ffsll((long long)e) - 1;
          upto = b == 63 ? ~0ull : ((2ull << b) - 1ull);
          nt_emit(p, s, __popcll(rest & upto));
          rest &= ~upto; e &= e - 1;
        }
        post = __popcll(rest);
      }
      // open bases arriving at each lane: scan of (has, value) with  (h1,v1) then (h2,v2) = (h1|h2, h2 ? v2 : v1+v2)
      uint32_t sh = has ? 1u : 0u, sv = has ? post : pre;
#pragma unroll
      for (int dd = 1; dd < 32; dd <<= 1) {
        const uint32_t oh = __shfl_up_sync(0xffffffffu, sh, dd), ov = __shfl_up_sync(0xffffffffu, sv, dd);
        if (lane >= dd) { sv = sh ? sv : ov + sv; sh |= oh; }
      }
      uint32_t eh = __shfl_up_sync(0xffffffffu, sh, 1), ev = __shfl_up_sync(0xffffffffu, sv, 1);   // exclusive
      if (lane == 0) { eh = 0; ev = 0; }
      const uint32_t open_in = eh ? ev : carry + ev;
      const bool is_head = has && !closed && !eh;               // the first run end of the piece: at most one lane
      if (has && !is_head) nt_emit(p, s, open_in + pre);
      const uint32_t head_src = __ballot_sync(0xffffffffu, is_head);
      if (head_src) head = __shfl_sync(0xffffffffu, open_in + pre, __ffs(head_src) - 1);
      const uint32_t th = __shfl_sync(0xffffffffu, sh, 31), tv = __shfl_sync(0xffffffffu, sv, 31);
      carry = th ? tv : carry + tv;
      closed = closed || th;
    }
    tail9 = __shfl_sync(0xffffffffu, (uint32_t)(m >> 55), 31);
    // every value read from the stage has been used: it can take the row NT_STAGES further on
    if (lane == 0 && k + NT_STAGES < n) {
      nt_issue(upcoming, ring + st * NT_STAGE, ring + NT_DESC_OFF + st * 16, ring + NT_BAR_OFF + st * 8);
      if (k + NT_STAGES + 1 < n) upcoming = mine[k + NT_STAGES + 1];
    }
    if (++st == NT_STAGES) { st = 0; phase ^= 1u; }
    if (last_row || k + 1 == n) {
      const uint32_t v[6] = {cA, cC, cG, cT, cN, cn};
#pragma unroll
      for (int i = 0; i < 6; ++i) { const uint32_t x = __reduce_add_sync(0xffffffffu, v[i]); if (lane == i && x) atomicAdd(&p.stats[(size_t)s * 8 + i], (unsigned long long)x); }
      if (lane == 0) { NtPiece r; r.head = head; r.tail = carry; r.closed = closed ? 1u : 0u; r.pad = 0; p.piece[(size_t)s + gw] = r; }
      cA = cC = cG = cT = cN = cn = 0; carry = 0; head = 0; closed = false;
    }
  }
}

}  // namespace

extern "C" {

// util/seqUtils.py:180-211 readFasta, as Python's text mode feeds it lines: "\n", "\r\n" and "\r" all end a line; lines that
// are blank after strip() are skipped; a header starts a record; of every other line the LAST CHARACTER IS DROPPED as its
// newline -- so a final line without one loses a base, as in the reference.
int ckm_fasta_scan_nt(const char *text, int64_t n, uint8_t *bytes_out, int64_t bytes_cap, int64_t *starts_out, int64_t *lens_out,
                      int32_t max_records, char *headers_out, int64_t headers_cap, int32_t *nrec_out, int64_t *bytes_used_out,
                      int64_t *hdr_bytes_out) {
  if ((!text && n > 0) || !bytes_out || !starts_out || !lens_out || !headers_out || !nrec_out || !bytes_used_out || !hdr_bytes_out) {
    set_error("ckm_fasta_scan_nt: bad argument"); return CKM_EINVAL;
  }
  int32_t nrec = 0; int64_t used = 0, hb = 0, i = 0;
  const bool has_cr = n > 0 && std::memchr(text, '\r', (size_t)n) != nullptr;      // files without one skip the per-line search
  auto close_record = [&]() {
    if (nrec == 0) return;
    const int64_t end = starts_out[nrec - 1] + lens_out[nrec - 1];
    const int64_t padded = (end + 63) / 64 * 64;
    std::memset(bytes_out + end, 0, (size_t)(padded - end));
    used = padded;
  };
  while (i < n) {
    const char *nl = (const char *)std::memchr(text + i, '\n', (size_t)(n - i));
    int64_t e = nl ? (nl - text) : n;                           // candidate line [i, e), terminator at e (or none)
    const char *cr = has_cr ? (const char *)std::memchr(text + i, '\r', (size_t)(e - i)) : nullptr;
    int64_t next = e + 1; bool terminated = nl != nullptr;
    if (cr) { e = cr - text; terminated = true; next = (e + 1 < n && text[e + 1] == '\n') ? e + 2 : e + 1; }
    bool blank = true;
    for (int64_t j = i; j < e && blank; ++j) { const unsigned char c = (unsigned char)text[j]; blank = (c == ' ' || (c >= 9 && c <= 13) || (c >= 28 && c <= 31)); }
    if (!blank) {
      if (text[i] == '>') {
        close_record();
        if (nrec >= max_records) { set_error("ckm_fasta_scan_nt: more records than the caller allowed for"); return CKM_ECAPACITY; }
        const int64_t len = e - (i + 1);
        if (hb + len + 1 > headers_cap) { set_error("ckm_fasta_scan_nt: header buffer too small"); return CKM_ECAPACITY; }
        if (nrec > 0) headers_out[hb++] = '\n';
        std::memcpy(headers_out + hb, text + i + 1, (size_t)len); hb += len;
        starts_out[nrec] = used; lens_out[nrec] = 0; ++nrec;
      } else {
        if (nrec == 0) { set_error("ckm_fasta_scan_nt: sequence data before the first '>' line"); return CKM_EFORMAT; }
        const int64_t len = terminated ? (e - i) : (e - i - 1);
        const int64_t at = starts_out[nrec - 1] + lens_out[nrec - 1];
        if (at + len + 64 > bytes_cap) { set_error("ckm_fasta_scan_nt: output buffer too small"); return CKM_ECAPACITY; }
        std::memcpy(bytes_out + at, text + i, (size_t)len);
        lens_out[nrec - 1] += len;
      }
    }
    i = next;
  }
  close_record();
  *nrec_out = nrec; *bytes_used_out = used; *hdr_bytes_out = hb;
  return CKM_OK;
}

int ckm_scaffold_stats(ckm_engine *e, const uint8_t *bytes, int64_t nbytes, const int64_t *starts, const int64_t *lens,
                       int32_t nscaf, int64_t *stats_out, uint32_t *contig_scaffold_out, uint32_t *contig_len_out,
                       int64_t contig_cap, int64_t *ncontigs_out, float *kernel_ms_out) {
  if (!e || nscaf < 0 || nbytes < 0 || (nscaf > 0 && (!bytes || !starts || !lens || !stats_out)) || contig_cap < 0 ||
      (contig_cap > 0 && (!contig_scaffold_out || !contig_len_out)) || !ncontigs_out) {
    set_error("ckm_scaffold_stats: bad argument"); return CKM_EINVAL;
  }
  *ncontigs_out = 0;
  if (kernel_ms_out) *kernel_ms_out = 0.0f;
  if (nscaf == 0) return CKM_OK;
  for (int32_t s = 0; s < nscaf; ++s) {
    if ((starts[s] & 63) || lens[s] < 0 || lens[s] > 0xFFFFFFFFll || starts[s] < 0 || (starts[s] + lens[s] + 63) / 64 * 64 > nbytes) {
      set_error("ckm_scaffold_stats: every scaffold must start at a multiple of 64 bytes and lie, padded to 64, inside the buffer");
      return CKM_EINVAL;
    }
  }
  cudaSetDevice(e->device);
  cudaStream_t st = e->stream;
  uint8_t *dbytes;
  int rc;
  if ((rc = workspace(e, Ws::NtBytes, (size_t)nbytes + 64, &dbytes))) return rc;
  std::vector<NtRow> rows;
  rows.reserve((size_t)(nbytes / NT_ROW) + nscaf);
  for (int32_t s = 0; s < nscaf; ++s)
    for (int64_t off = 0; off < lens[s]; off += NT_ROW) {
      const int64_t n = std::min<int64_t>(NT_ROW, lens[s] - off);
      const bool first = off == 0, last = off + NT_ROW >= lens[s];
      const int64_t left = first ? 0 : NT_HALO, copy = left + (n + 63) / 64 * 64 + (last ? 0 : NT_HALO);
      NtRow r; r.src = (uint64_t)(uintptr_t)(dbytes + starts[s] + off - left); r.scaf = (uint32_t)s;
      r.info = (uint32_t)n | ((uint32_t)(copy / 16) << 12) | (first ? 1u << 30 : 0u) | (last ? 1u << 31 : 0u);
      rows.push_back(r);
    }
  const int64_t nrows = (int64_t)rows.size();
  std::memset(stats_out, 0, sizeof(int64_t) * 8 * nscaf);
  if (nrows == 0) return CKM_OK;
  if (nrows > 0x7FFFFFFFll) { set_error("ckm_scaffold_stats: too many bytes for one call"); return CKM_EINVAL; }
  const int grid = (int)std::min<int64_t>((int64_t)e->prop.multiProcessorCount * NT_CTAS_PER_SM, (nrows + NT_WARPS - 1) / NT_WARPS);
  const int64_t nwarps = (int64_t)grid * NT_WARPS;
  const size_t npiece = (size_t)nscaf + nwarps;
  NtParams p;
  NtRow *drows; uint8_t *dctr;
  if ((rc = workspace(e, Ws::NtRows, sizeof(NtRow) * nrows, &drows)) || (rc = workspace(e, Ws::NtPieces, sizeof(NtPiece) * npiece, &p.piece)) ||
      (rc = workspace(e, Ws::NtStats, sizeof(int64_t) * 8 * nscaf, &p.stats)) ||
      (rc = workspace(e, Ws::NtContigScaf, sizeof(uint32_t) * (size_t)contig_cap, &p.contig_scaf)) ||
      (rc = workspace(e, Ws::NtContigLen, sizeof(uint32_t) * (size_t)contig_cap, &p.contig_len)) || (rc = workspace(e, Ws::NtCounters, 64, &dctr)))
    return rc;
  CKM_CUDA(cudaMemcpyAsync(dbytes, bytes, (size_t)nbytes, cudaMemcpyHostToDevice, st));
  CKM_CUDA(cudaMemcpyAsync(drows, rows.data(), sizeof(NtRow) * nrows, cudaMemcpyHostToDevice, st));
  CKM_CUDA(cudaMemsetAsync(p.piece, 0, sizeof(NtPiece) * npiece, st));
  CKM_CUDA(cudaMemsetAsync(dctr, 0, 64, st));
  CKM_CUDA(cudaMemsetAsync(p.stats, 0, sizeof(int64_t) * 8 * nscaf, st));
  p.bytes = dbytes; p.rows = drows; p.nrows = nrows;
  p.ncontigs = reinterpret_cast<unsigned long long *>(dctr + 8); p.cap = contig_cap;
  const int dyn_smem = NT_WARPS * NT_WARP_SMEM;
  CKM_CUDA(cudaFuncSetAttribute(ntstats_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, dyn_smem));
  CKM_CUDA(cudaEventRecord(e->ev[0], st));
  ntstats_kernel<<<grid, NT_THREADS, dyn_smem, st>>>(p);
  CKM_CUDA(cudaGetLastError());
  CKM_CUDA(cudaEventRecord(e->ev[1], st));
  unsigned long long n_dev = 0;
  std::vector<NtPiece> piece(npiece);
  CKM_CUDA(cudaMemcpyAsync(&n_dev, p.ncontigs, sizeof(n_dev), cudaMemcpyDeviceToHost, st));
  CKM_CUDA(cudaMemcpyAsync(stats_out, p.stats, sizeof(int64_t) * 8 * nscaf, cudaMemcpyDeviceToHost, st));
  CKM_CUDA(cudaMemcpyAsync(piece.data(), p.piece, sizeof(NtPiece) * npiece, cudaMemcpyDeviceToHost, st));
  CKM_CUDA(cudaStreamSynchronize(st));
  if (kernel_ms_out) CKM_CUDA(cudaEventElapsedTime(kernel_ms_out, e->ev[0], e->ev[1]));
  // join the open ends of the pieces, in list order: a contig runs from the tail of one piece through every piece without a
  // run end into the head of the next one of the same scaffold that has one
  std::vector<std::pair<uint32_t, uint32_t>> joined;
  {
    int64_t cur = -1; uint64_t open = 0;
    for (int64_t c = 0; c < nwarps; ++c) {
      const int64_t lo = nrows * c / nwarps, hi = nrows * (c + 1) / nwarps;
      if (lo >= hi) continue;
      for (int64_t s = rows[lo].scaf; s <= (int64_t)rows[hi - 1].scaf; ++s) {
        if (lens[s] == 0) continue;
        if (s != cur) { if (open) joined.emplace_back((uint32_t)cur, (uint32_t)open); cur = s; open = 0; }
        const NtPiece &r = piece[(size_t)s + c];
        if (r.closed) { if (open + r.head) joined.emplace_back((uint32_t)s, (uint32_t)(open + r.head)); open = r.tail; }
        else open += r.tail;
      }
    }
    if (open) joined.emplace_back((uint32_t)cur, (uint32_t)open);
  }
  const int64_t n_found = (int64_t)n_dev + (int64_t)joined.size();
  *ncontigs_out = n_found;
  if (n_found > contig_cap) { set_error("ckm_scaffold_stats: more contigs than the caller allowed for (the count is returned; call again)"); return CKM_ECAPACITY; }
  if (n_dev) {
    CKM_CUDA(cudaMemcpyAsync(contig_scaffold_out, p.contig_scaf, sizeof(uint32_t) * n_dev, cudaMemcpyDeviceToHost, st));
    CKM_CUDA(cudaMemcpyAsync(contig_len_out, p.contig_len, sizeof(uint32_t) * n_dev, cudaMemcpyDeviceToHost, st));
    CKM_CUDA(cudaStreamSynchronize(st));
  }
  for (size_t k = 0; k < joined.size(); ++k) {
    contig_scaffold_out[n_dev + k] = joined[k].first; contig_len_out[n_dev + k] = joined[k].second;
    stats_out[(size_t)joined[k].first * 8 + 6] += 1; stats_out[(size_t)joined[k].first * 8 + 7] += joined[k].second;
  }
  return CKM_OK;
}

}  // extern "C"
