/*
 * ckm.h -- C-ABI of libckm.so, the B200-native marker-gene search engine behind CheckM's
 * HMMERRunner / MarkerGeneFinder / ResultsParser surfaces.
 *
 * The reference has no FFI on this path: it crosses a process + text-file boundary,
 *     os.system('hmmsearch --domtblout T opts HMM FAA > OUT')            (checkm/hmmer.py:70-71)
 *     os.system('hmmfetch -f db keyfile > out'), 'hmmfetch --index'      (checkm/hmmer.py:107,126)
 * and re-parses the text (checkm/hmmer.py:184-200) before the Python reduction
 * (checkm/resultsParser.py:340-479,513-537; checkm/util/pfam.py:86-147; checkm/markerSets.py:206-238).
 * Each entry point below names the reference interface it replaces.  INTEGRATION.md shows the ctypes
 * binding a CheckM maintainer would add.
 *
 * Conventions: every function returns 0 on success and a non-zero ckm_status otherwise (the Python shim
 * maps that to logger.error + sys.exit(rtn), mirroring checkm/hmmer.py:72-74); ckm_last_error() gives the
 * message.  Plain pointers and sizes only.  Inputs are borrowed for the duration of the call; outputs are
 * owned by the library until the matching *_free.  One engine per process per GPU; not thread-safe; a
 * CUDA context cannot cross fork(), so create the engine in the process that uses it.
 * There is no CPU fallback: without a CUDA device ckm_init fails with CKM_ENODEVICE.
 */
#ifndef CKM_H
#define CKM_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
  CKM_OK = 0,
  CKM_EINVAL = 1,      /* bad argument                                   */
  CKM_EIO = 2,         /* cannot open / write a file                     */
  CKM_EFORMAT = 3,     /* malformed HMMER3/f file                        */
  CKM_ENODEVICE = 4,   /* no usable CUDA device                          */
  CKM_ECUDA = 5,       /* CUDA runtime error                             */
  CKM_ENOMEM = 6,
  CKM_ENOTFOUND = 7,   /* accession / name not in the model database     */
  CKM_ECAPACITY = 8    /* an internal device queue overflowed            */
} ckm_status;

typedef struct ckm_engine   ckm_engine;
typedef struct ckm_models   ckm_models;    /* a parsed + configured HMM database, resident on the device */
typedef struct ckm_seqdb    ckm_seqdb;     /* digitised ORFs of one or more bins, resident on the device  */

/* ---- header fields CheckM reads from a model (checkm/hmmerModelParser.py:27-83) ---- */
typedef struct {
  char   name[128];
  char   acc[64];       /* empty string when the model has no ACC line */
  char   desc[256];
  int32_t M;            /* LENG */
  int32_t has_ga, has_tc, has_nc;
  float  ga[2], tc[2], nc[2];
  float  evparam[6];    /* MSV mu, lambda; VITERBI mu, lambda; FORWARD tau, lambda */
  double ga_d[2], tc_d[2], nc_d[2];   /* the cutoffs as Python's float() reads the header text (hmmerModelParser.py:76) */
} ckm_model_info;

/* ---- one reported domain = one domtblout row (checkm/hmmer.py:255-285 field for field) ---- */
typedef struct {
  int32_t bin;          /* index into the bins of the seqdb                                  */
  int32_t seq;          /* target: global sequence index in the seqdb   (target_name)        */
  int32_t model;        /* query: model index in the ckm_models          (query_name/acc)     */
  int32_t tlen;         /* target_length (residues incl. trailing '*')                       */
  int32_t qlen;         /* query_length  (model length M)                                    */
  int32_t dom, ndom;    /* '#' and 'of'                                                      */
  int32_t hmm_from, hmm_to, ali_from, ali_to, env_from, env_to;
  float   full_score, full_bias;    /* bits                                                  */
  float   dom_score, dom_bias;      /* bits                                                  */
  float   acc;                      /* mean posterior of the aligned residues                */
  double  full_evalue, c_evalue, i_evalue;
  double  full_lnP, dom_lnP;        /* natural-log P-values before multiplying by Z / domZ   */
} ckm_hit;

/* ---- counters of the filter cascade, for tests and profiling ---- */
typedef struct {
  int64_t n_pairs;        /* (ORF x HMM) pairs scored by the SSV/MSV stage    */
  int64_t n_cells;        /* sum of L*M over those pairs                      */
  int64_t n_ssv_cand;     /* pairs the SSV pre-filter fires on (scored exactly, in its epilogue or by the exact MSV kernels) */
  int64_t n_past_msv, n_past_bias, n_past_vit, n_past_fwd;
  int64_t n_hits_seq;     /* targets in the hit list (before E thresholds)    */
  int64_t n_domains;      /* domains defined                                  */
  int64_t n_reported;     /* domtblout rows                                   */
  float   ms_ssv, ms_msv, ms_bias, ms_vit, ms_fwd, ms_domdef, ms_total;   /* CUDA-event times of the last search */
  int64_t kernel_launches;
  int64_t n_vit_redo;     /* pairs the packed Viterbi kernel handed to the int32 kernel (strong hits, guard conditions) */
  int64_t n_msv_exact;    /* of n_ssv_cand, the pairs forwarded to the exact MSV kernels (J-eligible, capped, chained) */
  int64_t n_queue_retries;/* times the filter cascade was re-run with larger candidate queues (candidate-dense input) */
} ckm_stats;

/* ---- per-bin QA row = the integers/floats behind CheckM's table
 *      (checkm/resultsParser.py:513-537 geneCounts; checkm/markerSets.py:206-238 genomeCheck) ---- */
typedef struct {
  int32_t bin;
  int32_t counts[6];          /* markers found 0,1,2,3,4,5+ times                 */
  int32_t n_markers, n_sets;
  int32_t unique_hits, multi_hits;   /* countUniqueHits (resultsParser.py:481-491) */
  double  completeness, contamination;
} ckm_qa_row;

/* ---- one surviving marker hit after the reduction (an element of ResultsManager.markerHits[acc]) ---- */
typedef struct {
  int32_t bin, model;
  int32_t seq_a, seq_b;       /* seq_b >= 0 for an adjacent-ORF merge: name is "A&&B" with A < B (string order) */
  int32_t target_length;
  int32_t hmm_from, hmm_to, ali_from, ali_to, env_from, env_to;
  int32_t order;              /* position within markerHits[acc] for this bin                               */
  int32_t src_row;            /* index of the ckm_hit row that carries this hit's scores / E-values        */
  int64_t dict_key;           /* orders the markers of a bin as the reference's markerHits dict iterates them:
                                 -1 for non-Pfam markers (they keep file order and come first, pfam.py:93-100), else the
                                 position at which the clan filter re-inserted the marker (pfam.py:141-145)       */
} ckm_marker_hit;

/* ---- lifecycle ---- */
int  ckm_init(int device, ckm_engine **out);                     /* replaces HMMERRunner.checkForHMMER (hmmer.py:131-137) */
void ckm_destroy(ckm_engine *e);
const char *ckm_last_error(void);
const char *ckm_version(void);
int  ckm_device_name(ckm_engine *e, char *buf, int buflen);

/* ---- models: parse HMMER3/f (header AND body), configure MSV/Viterbi/Forward profiles, upload ----
 * replaces hmmsearch's own reading of <hmmfile> and HmmModelParser.simpleParse (hmmerModelParser.py:46-83).
 * A model may have up to 4,608 match positions (the DP rows of the chunked kernels live in shared memory); a longer one makes
 * the call fail with CKM_EINVAL and the model's name in ckm_last_error().  Models of 3,072 positions and more are searched
 * without the SSV pre-filter (same results, every pair scored by the exact MSV kernel). */
int  ckm_models_load(ckm_engine *e, const char *hmm_path, ckm_models **out);
int  ckm_models_count(const ckm_models *m);
int  ckm_models_info(const ckm_models *m, int idx, ckm_model_info *out);
int  ckm_models_find(const ckm_models *m, const char *key);      /* by accession or name; -1 if absent */
/* subset by accession/name list, in database order: replaces `hmmfetch -f` + `hmmfetch --index`
 * (checkm/markerSets.py:443-476, checkm/hmmer.py:97-129).  idx_out[n] receives database indices. */
int  ckm_models_select(const ckm_models *m, const char *const *keys, int nkeys, int32_t *idx_out, int *n_out);
/* write the selected models back out as a HMMER3/f file (what `hmmfetch -f db keys > out` produced) */
int  ckm_models_write(const ckm_models *m, const int32_t *idx, int n, const char *out_path);
void ckm_models_free(ckm_models *m);

/* ---- sequences: digitised residues (codes 0..28 of "ACDEFGHIKLMNPQRSTVWY-BJZOUX*~"), CSR offsets,
 *      bin id per sequence.  Replaces hmmsearch's reading of <seqfile> (genes.faa). ---- */
int  ckm_digitize(const char *text, int64_t n, uint8_t *out);    /* ASCII -> codes; returns #unknown symbols via negative? no: 0 */
/* a whole protein FASTA file (genes.faa, checkm/markerGeneFinder.py:113-127) in one pass: residue codes, CSR offsets
 * (max_records + 1 entries) and the header lines (text after '>', joined by '\n') from which the caller takes names and
 * descriptions.  residues_out needs n bytes, headers_out at most n. */
int  ckm_fasta_parse(const char *text, int64_t n, uint8_t *residues_out, int64_t *offsets_out, int32_t max_records,
                     char *headers_out, int64_t headers_cap, int32_t *nrec_out, int64_t *nres_out, int64_t *hdr_bytes_out);
int  ckm_seqdb_create(ckm_engine *e, const uint8_t *residues, const int64_t *seq_offsets, int32_t nseq,
                      const int32_t *bin_of_seq, int32_t nbins, ckm_seqdb **out);
void ckm_seqdb_free(ckm_seqdb *db);

/* ---- the search: MSV -> bias -> Viterbi -> Forward -> domain definition -> E-values / thresholds.
 * replaces HMMERRunner.search = os.system('hmmsearch --domtblout ...') (checkm/hmmer.py:61-74) with the
 * options CheckM passes (markerGeneFinder.py:141): -E <E> --domE <domE>; Z = #sequences of the bin.
 * model_idx selects the queries (NULL = all).  Rows come back grouped by bin, then by query in the order
 * given, then by target E-value -- the order hmmsearch writes them. */
int  ckm_search(ckm_engine *e, const ckm_models *m, const int32_t *model_idx, int32_t nmodels,
                const ckm_seqdb *db, double E, double domE, ckm_hit **hits_out, int64_t *nhits_out);
/* same, with per-bin query subsets (lineage_wf: every bin has its own marker HMMs): CSR over bins */
int  ckm_search_per_bin(ckm_engine *e, const ckm_models *m, const int32_t *model_idx, const int64_t *bin_model_offsets,
                        const ckm_seqdb *db, double E, double domE, ckm_hit **hits_out, int64_t *nhits_out);
void ckm_hits_free(ckm_hit *hits);

/* ---- hmmalign: optimal-accuracy alignment of every sequence of `db` to ONE model, configured as `hmmalign` does (unihit
 * local; Forward, Backward, posterior decoding, optimal-accuracy fill + traceback over the whole sequence).
 * replaces HMMERRunner.align = os.system('hmmalign --outformat ... db query > out') (checkm/hmmer.py:76-95), whose output
 * CheckM masks down to the match columns (checkm/hmmerAligner.py:276-358).
 * state_out[r] for residue r of the unpadded stream (ckm_seqdb_create offsets): k > 0 emitted by match state k, k < 0 by
 * insert state -k, 0 unaligned flank.  oasc_out[nseq] (optional): the optimal-accuracy score, 0 if no alignment exists. ---- */
int  ckm_align(ckm_engine *e, const ckm_models *m, int32_t model, const ckm_seqdb *db, int32_t *state_out, float *oasc_out);
int  ckm_last_stats(const ckm_engine *e, ckm_stats *out);
/* device bytes the engine keeps between calls as workspaces (one grow-only buffer per role, slack included); models, sequence
 * databases and the stream-ordered pool are not counted.  It follows from the largest inputs the engine has seen, not from
 * the order of its calls. */
int  ckm_workspace_bytes(const ckm_engine *e, int64_t *bytes_out);

/* stage-level entry points for parity tests (device arrays come back to host buffers the caller owns) */
int  ckm_msv_scores(ckm_engine *e, const ckm_models *m, const int32_t *model_idx, int32_t nmodels,
                    const ckm_seqdb *db, int32_t *xj_out /* nmodels*nseq; 256 = overflow; -1 = not a candidate */);
int  ckm_filter_scores(ckm_engine *e, const ckm_models *m, const int32_t *model_idx, int32_t nmodels,
                       const ckm_seqdb *db, float *filtersc_out, float *vit_out, float *fwd_out,
                       uint8_t *passed_out /* bit0 msv, bit1 bias, bit2 vit, bit3 fwd; each nmodels*nseq */);

/* ViterbiFilter score (nats) of EVERY pair, through the production kernels: the packed int16x2 kernel with its int32
 * redo list (mode 0), the int32 kernels alone (mode 1), or the chunked shared-memory int32 kernel for every model, which
 * production uses only beyond M = 1024 (mode 2).  +inf = int16 overflow, -inf = no path.  n_vit_redo of
 * ckm_last_stats says how many pairs took the redo route. */
int  ckm_viterbi_scores(ckm_engine *e, const ckm_models *m, const int32_t *model_idx, int32_t nmodels,
                        const ckm_seqdb *db, int32_t mode, float *vit_out /* nmodels*nseq */);

/* ---- domtblout text for one bin of a finished search: the file CheckM's HMMERParser re-reads
 * (checkm/hmmer.py:184-200).  names/descs are the FASTA header words of the bin's sequences. ---- */
int  ckm_write_domtblout(const ckm_models *m, const ckm_hit *hits, int64_t nhits, int32_t bin,
                         int32_t seq_base, const char *const *names, const char *const *descs, const char *path);

/* ---- the reduction: vetHit -> addHit -> PFAM clan filter -> adjacent-ORF merge -> gene counts ->
 * completeness / contamination, on the device, for every bin of a finished search.
 * replaces ResultsParser.parseBinHits + ResultsManager.* + PFAM.filterHitsFromSameClan + MarkerSet.genomeCheck
 * (checkm/resultsParser.py:76-119,340-479,481-537; checkm/util/pfam.py:86-147; checkm/markerSets.py:206-238). */
typedef struct {
  int32_t ignore_thresholds;        /* bIgnoreThresholds                                   */
  int32_t skip_pseudogene;          /* bSkipPseudoGeneCorrection                           */
  int32_t skip_adjacent;            /* bSkipAdjCorrection                                  */
  int32_t individual_markers;       /* bIndividualMarkers                                  */
  double  evalue_threshold;         /* DefaultValues.E_VAL = 1e-10                         */
  int32_t evalue_exp10;             /* the same threshold as mant x 10^(exp10-1), 10 <= mant < 100, decomposed */
  int32_t pad0;                     /*   exactly (decimal) by the caller: the reference compares the 2-digit    */
  double  evalue_mant;              /*   text of the E-value (hmmer.py:268) against it                         */
  double  length_threshold;         /* DefaultValues.LENGTH = 0.7                          */
  double  pseudogene_length;        /* DefaultValues.PSEUDOGENE_LENGTH = 0.3               */
} ckm_reduce_opts;

/* Per-model reduction metadata derived on the host from names / Pfam-A.hmm.dat (pfam.py:34-56):
 *   is_pfam[m]   marker id starts with "PF"
 *   is_tigr[m]   'TIGR' in accession                                  (resultsParser.py:356)
 *   clan[m]      clan id (>=0) or -1; two clan-less Pfams compare equal, as in the reference (pfam.py:131)
 *   nest_off/nest_idx: CSR of model indices nested with m             (pfam.py:48-56)
 * Per-sequence metadata from the ORF names (resultsParser.py:411-427):
 *   scaffold_id[s] integer id of name[:rfind('_')], orf_num[s] int(name[rfind('_')+1:]) or INT32_MIN if not an int
 * Marker sets per bin (markerSets.py:206-238): CSR bin -> sets -> model indices.
 * The printed/rounded score and E-value columns are what the reference compares (hmmer.py:269-276), so the
 * reduction rounds full_score/dom_score to %.1f and E-values to %.2g exactly as the text round trip does. */
typedef struct {
  const uint8_t *is_pfam, *is_tigr;
  const int32_t *clan;
  const int64_t *nest_off; const int32_t *nest_idx;
  const int32_t *has_cut;                        /* nmodels x {ga, tc, nc}: cutoff present                          */
  const double  *cutoffs;                        /* nmodels x {ga0, ga1, tc0, tc1, nc0, nc1} as float() reads them  */
  const double  *row_scores;                     /* optional, nhits x {full_score, dom_score}: the values exactly as the
                                                    domtblout text gave them (text path); NULL = round the binary scores to %.1f */
  const int32_t *scaffold_id, *orf_num;          /* per sequence */
  const int32_t *name_rank;                      /* per sequence: rank of the name in string order (for "A&&B") */
  const int64_t *bin_set_off;                    /* optional: nbins+1; sets of bin b are [bin_set_off[b], bin_set_off[b+1]) */
  const int64_t *set_marker_off;                 /* nsets+1 */
  const int32_t *set_marker_idx;                 /* model indices */
} ckm_reduce_meta;

/* hits: domtblout rows grouped by bin (ascending) and, inside a bin, by query (rows of one query contiguous, in file
 * order).  `model` and `seq` index the caller's model table (nmodels entries) and sequence table (nseq entries).
 * When the device has no room left for the reduction, the engine's workspaces (ckm_workspace_bytes) are freed and the call
 * is tried once more; the engine's next call allocates what it needs again. */
int  ckm_reduce(ckm_engine *e, int32_t nmodels, int32_t nseq, int32_t nbins, const ckm_hit *hits, int64_t nhits,
                const ckm_reduce_opts *opts, const ckm_reduce_meta *meta,
                ckm_qa_row **qa_out, int32_t *nqa_out, ckm_marker_hit **mh_out, int64_t *nmh_out);
/* completeness / contamination / copy-number histogram from per-marker copy numbers, on the device
 * (ResultsManager.geneCounts + MarkerSet.genomeCheck for an arbitrary {marker: hits} dict, e.g. merger.py:63-88).
 * marker_count[y] is the copy number of the y-th entry of the sets CSR. */
int  ckm_genome_check(ckm_engine *e, int32_t nbins, const int64_t *bin_set_off, const int64_t *set_marker_off,
                      const int32_t *marker_count, int32_t individual_markers, ckm_qa_row *rows_out);
void ckm_free(void *p);

/* ---- multi-GPU (SURVEY.md 8e; BASELINE.json configs[3] "NCCL gather of qa table"): bins are sharded over ranks, one
 * process per GPU; the only inter-GPU traffic is one ncclAllGather of the fixed-width QA rows.  The communicator is the
 * caller's (an ncclComm_t from ncclCommInitRank) or one made here: rank 0 calls ckm_nccl_unique_id, ships the 128 bytes to
 * the other ranks by whatever channel it has (MPI, torch.distributed, a file), every rank calls ckm_nccl_comm_init.
 * rows_out holds world * nrows_max rows (rank r's rows start at r * nrows_max), counts_out the row count of every rank. ---- */
int  ckm_nccl_unique_id(uint8_t *id_out, int32_t nbytes);
int  ckm_nccl_comm_init(ckm_engine *e, int32_t world, int32_t rank, const uint8_t *id, void **comm_out);
void ckm_nccl_comm_destroy(void *comm);
int  ckm_allgather_qa(ckm_engine *e, void *nccl_comm, const ckm_qa_row *rows, int32_t nrows, int32_t nrows_max,
                      int32_t world, ckm_qa_row *rows_out, int32_t *counts_out);

/* ---- bin statistics (SURVEY.md 8 row f4; checkm/binStatistics.py:99-139,176-243): the integer half -- base counts,
 * ambiguous bases and the contig lengths of every scaffold -- as one byte scan on the device; the caller forms GC, N50 and
 * the means from these integers exactly as the reference does from its own counts. ---- */
/* a nucleotide FASTA file read the way checkm/util/seqUtils.py:180-211 readFasta reads it (text-mode line ends, blank lines
 * skipped, the last character of a final unterminated line lost).  Record r occupies bytes_out[starts_out[r] ..
 * starts_out[r] + lens_out[r]), starts are multiples of 64 and the gaps are zero: the layout ckm_scaffold_stats wants.
 * bytes_cap >= n + 64 * (max_records + 1) always suffices.  Header lines come back as in ckm_fasta_parse. */
int  ckm_fasta_scan_nt(const char *text, int64_t n, uint8_t *bytes_out, int64_t bytes_cap, int64_t *starts_out, int64_t *lens_out,
                       int32_t max_records, char *headers_out, int64_t headers_cap, int32_t *nrec_out, int64_t *bytes_used_out,
                       int64_t *hdr_bytes_out);
/* stats_out: nscaf x 8 int64 = {A, C, G, T+U (all case-insensitive, seqUtils.py:279-286), 'N', 'n', contigs, contig bases};
 * a contig is a stretch between runs of >= 10 'N' (DefaultValues.CONTIG_BREAK), its length the bytes in it that are not 'N'
 * (binStatistics.py:208-226).  The contigs of all scaffolds come back as (scaffold, length) pairs in no particular order;
 * with more than contig_cap of them the call fails with CKM_ECAPACITY and *ncontigs_out holds the number needed.
 * kernel_ms_out (optional): duration of the scan kernel by CUDA events. */
int  ckm_scaffold_stats(ckm_engine *e, const uint8_t *bytes, int64_t nbytes, const int64_t *starts, const int64_t *lens,
                        int32_t nscaf, int64_t *stats_out, uint32_t *contig_scaffold_out, uint32_t *contig_len_out,
                        int64_t contig_cap, int64_t *ncontigs_out, float *kernel_ms_out);

#ifdef __cplusplus
}
#endif
#endif
