/* kaiju_b200.h -- C ABI of the B200-native Kaiju classification path (libkaijub200.so).
 *
 * Drop-in boundary: the reference has no FFI; its seam is the C++ class ConsumerThread
 * (src/ConsumerThread.hpp:64-121): N threads each pop ReadItem* from a queue, classify it against the
 * shared read-only Config (FMI + suffix array + nodes map) and append "C\tname\ttaxid\n" lines.  This
 * library replaces everything between "ReadItems popped" and "taxon id known" for a whole batch:
 *
 *   reference call / type                                    replaced by
 *   -------------------------------------------------------  -------------------------------------
 *   readFMI + Config::init        (util.cpp:265-276, Config.cpp:19-28)   kj_index_view (views into the loader's
 *                                                                         buffers) or kj_fmi_load() (our loader)
 *   parseNodesDmp                 (util.cpp:79-99)                        kj_taxonomy_view or kj_nodes_load()
 *   new ConsumerThread(queue,config) x N (kaiju.cpp:250-257)              kj_create()
 *   ConsumerThread::doWork        (ConsumerThread.cpp:630-749)            kj_classify() / kj_classify_device()
 *   delete ConsumerThread / Config                                         kj_destroy()
 *
 * All entry points return 0 on success or a negative kj_status; the library never calls exit().
 * Plain pointers and sizes only; the caller owns every buffer it passes in.
 */
#ifndef KAIJU_B200_H
#define KAIJU_B200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
    KJ_OK = 0,
    KJ_ERR_ARG = -1,            /* null/invalid argument */
    KJ_ERR_IO = -2,             /* file could not be read / is not a .fmi */
    KJ_ERR_CUDA = -3,           /* CUDA runtime failure (kj_last_error() has the text) */
    KJ_ERR_NO_DEVICE = -4,      /* no usable GPU: there is NO CPU fallback */
    KJ_ERR_UNSUPPORTED = -5,    /* alphabet > 24 letters, read longer than KJ_MAX_READ_LEN, -e > 8 ... */
    KJ_ERR_OVERFLOW = -6,       /* an internal per-read work queue overflowed (results of the batch are invalid) */
    KJ_ERR_NOMEM = -7
} kj_status;

#define KJ_MAX_READ_LEN 16383   /* bases per mate (queue payloads carry 15-bit array positions; fragment scores stay below 2^16) */
#define KJ_MAX_PROTEIN_LEN 5461 /* residues of a protein read (-p): stored like one reading frame of a KJ_MAX_READ_LEN read */

/* Mode / Config fields consumed by the path (src/Config.hpp:31-66, set by kaiju.cpp:74-202) */
typedef struct {
    int32_t mode;                 /* 0 = MEM (-a mem), 1 = GREEDY (-a greedy)            */
    uint32_t min_fragment_length; /* -m, default 11                                      */
    uint32_t mismatches;          /* -e, default 3  (Greedy)                             */
    uint32_t min_score;           /* -s, default 65 (Greedy)                             */
    uint32_t seed_length;         /* -l, default 7  (Greedy)                             */
    int32_t use_evalue;           /* Greedy: 1 unless disabled; MEM: must be 0           */
    double min_evalue;            /* -E, default 0.01                                    */
    int32_t seg;                  /* -x (1, default) / -X (0)                            */
    int32_t input_is_protein;     /* -p: seq1 holds protein letters, seq2 must be NULL  */
    int32_t name_mode;            /* 1: search as the kaijux / kaijup front-ends do (ConsumerThreadx.cpp:117-190): MEM keeps the matches of a
                                     fragment in maxMatches order (bwt.c:225-296) instead of greedyExact order; Greedy is unchanged.
                                     The caller passes an index view whose seq_taxon numbers the sequences (see INTEGRATION.md 2d). */
} kj_params;

/* Host views straight out of a .fmi loader (the reference's BWT/FMI/suffixArray structs:
 * bwt/bwt.h:13-23, bwt/compactfmi.h:10-19, bwt/suffixArray.h:10-33).  Nothing is retained after kj_create(). */
typedef struct {
    int32_t alen;                 /* FMI.alen (alphabet incl. terminator, 21 for proteins)          */
    const char *alphabet;         /* BWT.alphabet ("*ACDEFGHIKLMNPQRSTVWY")                         */
    int64_t bwtlen;               /* FMI.bwtlen                                                      */
    const uint8_t *bwt;           /* FMI.bwt : byte codes (letter + distance), length bwtlen         */
    const int32_t *startLcode;    /* FMI.startLcode[alen+1] : code range of each letter              */
    int64_t db_len;               /* BWT.len  (E-value uses len - nseq, Config.cpp:20)               */
    int32_t nseq;                 /* BWT.nseq                                                        */
    int64_t ncheck;               /* suffixArray.ncheck                                              */
    int32_t chpt_exp, nbytes, pbits; /* suffixArray.chpt_exp / nbytes / pbits                        */
    const uint8_t *sa;            /* suffixArray.sa : ncheck * nbytes big-endian packed (seq,pos)     */
    const uint64_t *seq_taxon;    /* [nseq] taxon id parsed from suffixArray.ids[i] with the rule of
                                     ConsumerThread.cpp:812-832 (UINT64_MAX = "bad number", skipped) */
    const uint32_t *seq_accession;/* optional [nseq] (NULL = not given): rank of the sequence's accession -- its name up to the last '_' --
                                     among the distinct accessions in lexicographic order, 0xffffffff for names without '_'
                                     (ConsumerThread.cpp:809-823); only kj_classify_verbose2() needs it (column 6 of `kaiju -v`) */
} kj_index_view;

typedef struct {
    uint64_t n;                   /* number of (node,parent) pairs, i.e. nodes.dmp lines             */
    const uint64_t *node;         /* child taxon id                                                   */
    const uint64_t *parent;       /* parent taxon id (root: parent == node)                           */
} kj_taxonomy_view;

typedef struct kj_fmi kj_fmi;           /* an owned, parsed .fmi file                */
typedef struct kj_nodes kj_nodes;       /* an owned, parsed nodes.dmp                */
typedef struct kj_ctx kj_ctx;           /* one GPU context: index + taxonomy in HBM  */

/* --- loaders (our own re-implementation of the on-disk formats; SURVEY.md 8a row 14) --- */
int kj_fmi_load(const char *path, kj_fmi **out);
void kj_fmi_view(const kj_fmi *f, kj_index_view *view);
void kj_fmi_free(kj_fmi *f);
const char *kj_fmi_seq_name(const kj_fmi *f, int32_t i);
/* accession ranks of the sequences (what kj_index_view.seq_accession takes; kj_fmi_view() fills it in) and the accession string of a rank */
const char *kj_fmi_accession(const kj_fmi *f, uint32_t rank);   /* suffixArray.ids[i]: the database name of sequence i (in the index's own order) */
int kj_nodes_load(const char *path, kj_nodes **out);
void kj_nodes_view(const kj_nodes *t, kj_taxonomy_view *view);
void kj_nodes_free(kj_nodes *t);

/* --- context --- */
/* Transcodes the index into the device layout, uploads it and the taxonomy to HBM of `device`. */
int kj_create(kj_ctx **out, int device, const kj_params *params, const kj_index_view *index, const kj_taxonomy_view *taxonomy);
/* The large arrays (rank records, packed letters, taxon-reduced suffix array, k-mer table) are built ON THE DEVICE from the raw BWT bytes and
 * suffix-array samples of the view (SURVEY.md 8f-4; replaces the table construction of mkfmi.c:63-78 / fmicommon.h:104-184).
 * kj_create_scaled: the index of the collection in which every sequence of `index` occurs `copies` times in a row -- identical to what
 * kaiju-mkbwt/-mkfmi produce for the K-fold FASTA (identical suffixes are ordered by sequence number), derived on the device without a
 * suffix sort.  With all copies carrying the taxon of their original, MEM results equal those on the base index; it exists to bring
 * refseq_ref-scale indexes (2.7e10 rows, ~126 GB in HBM) onto a GPU for capacity and throughput measurements.  copies = 1 == kj_create. */
int kj_create_scaled(kj_ctx **out, int device, const kj_params *params, const kj_index_view *index, const kj_taxonomy_view *taxonomy, uint32_t copies);
double kj_index_build_ms(const kj_ctx *ctx);      /* wall time of the index construction inside kj_create / kj_create_scaled */
/* Device-native index file (SURVEY.md 8f-4): kj_native_index_write() transcodes once (the .fmi + nodes.dmp views as for kj_create) and
 * stores the arrays exactly as they are uploaded (one-hot rank records, packed letters, taxon-reduced suffix array, re-indexed
 * taxonomy, k-mer table); kj_create_from_native() then needs one sequential read and the upload -- no transcode at load time.
 * The file is specific to this library version (checked; KJ_ERR_IO otherwise). */
int kj_native_index_write(const kj_index_view *index, const kj_taxonomy_view *taxonomy, const char *path);
int kj_create_from_native(kj_ctx **out, int device, const kj_params *params, const char *path);
/* Change the run parameters of an existing context (index stays resident). */
int kj_set_params(kj_ctx *ctx, const kj_params *params);
void kj_destroy(kj_ctx *ctx);

/* --- classification --- */
/* Host buffers.  seq1 = concatenated bases of mate 1, off1[n_reads+1] byte offsets; seq2/off2 = mate 2 or NULL
 * for single-end input.  taxon_out[n_reads]: NCBI taxon id, 0 = unclassified (the "U" line).  best_out (optional):
 * match length (MEM) or score (Greedy) -- column 4 of the reference's -v output.  Blocking; H2D/D2H inside. */
int kj_classify(kj_ctx *ctx, const char *seq1, const uint64_t *off1, const char *seq2, const uint64_t *off2,
                uint64_t n_reads, uint64_t *taxon_out, uint32_t *best_out);
/* Same, plus column 5 of the reference's -v output (ConsumerThread.cpp:527-536, 614-623): the match-id set of every classified read,
 * ascending, ids_out[i*KJ_MAX_MATCH_IDS .. +nids_out[i]) (at most 21 ids: max_match_ids = 20 is checked before each insertion). */
#define KJ_MAX_MATCH_IDS 21
int kj_classify_verbose(kj_ctx *ctx, const char *seq1, const uint64_t *off1, const char *seq2, const uint64_t *off2,
                        uint64_t n_reads, uint64_t *taxon_out, uint32_t *best_out, uint64_t *ids_out, uint8_t *nids_out);
/* All seven columns of `kaiju -v` (ConsumerThread.cpp:527-536, 614-623): additionally the accession set of the visited database sequences
 * (acc_out[i*KJ_MAX_MATCH_ACC .. +nacc_out[i]), ranks as given in kj_index_view.seq_accession, ascending = the reference's std::set<string>
 * order; the context must have been created from a view with seq_accession) and the matched fragment strings, ready to print
 * ("IGEYVEMMNGVVLSYIES,..." in frag_out[i*frag_stride .. +frag_len_out[i])): MEM = the longest match of every fragment that reached the
 * longest length, Greedy = the sequences (with substitutions) of the best matches.  A read whose strings exceed frag_stride bytes makes the
 * call fail with KJ_ERR_OVERFLOW. */
#define KJ_MAX_MATCH_ACC 20
int kj_classify_verbose2(kj_ctx *ctx, const char *seq1, const uint64_t *off1, const char *seq2, const uint64_t *off2,
                         uint64_t n_reads, uint64_t *taxon_out, uint32_t *best_out, uint64_t *ids_out, uint8_t *nids_out,
                         uint32_t *acc_out, uint8_t *nacc_out, char *frag_out, uint32_t frag_stride, uint32_t *frag_len_out);
/* With params.input_is_protein (-p) seq1 holds protein letters (split at every letter outside the 20 residues,
 * ConsumerThread.cpp:659-696) and seq2 must be NULL.  Reads longer than KJ_MAX_READ_LEN / KJ_MAX_PROTEIN_LEN -> KJ_ERR_UNSUPPORTED. */
/* Device buffers (same layout, all pointers in the context's device memory), enqueued on `cuda_stream`
 * (a cudaStream_t, NULL = default stream); returns after the launch, results are ready when the stream is.
 * max_len1/max_len2: upper bounds of the mate lengths in the batch (0 = let the library compute them on the device). */
int kj_classify_device(kj_ctx *ctx, const char *d_seq1, const uint64_t *d_off1, const char *d_seq2, const uint64_t *d_off2,
                       uint64_t n_reads, uint32_t max_len1, uint32_t max_len2, uint64_t *d_taxon_out, uint32_t *d_best_out,
                       void *cuda_stream);

/* Variants with a DEVICE array d_compact_out[n_reads] (optional, may be NULL): the dense taxon index of every read as uint32 (position of
 * the taxon in kj_counts_get()'s id list, 0xffffffff = unclassified) -- what the ranks of a multi-GPU job all-gather instead of the
 * 64-bit NCBI ids (SURVEY.md 8e).  kj_classify_device2 accepts d_taxon_out == NULL when d_compact_out is given. */
int kj_classify2(kj_ctx *ctx, const char *seq1, const uint64_t *off1, const char *seq2, const uint64_t *off2,
                 uint64_t n_reads, uint64_t *taxon_out, uint32_t *best_out, uint32_t *d_compact_out);
int kj_classify_device2(kj_ctx *ctx, const char *d_seq1, const uint64_t *d_off1, const char *d_seq2, const uint64_t *d_off2,
                        uint64_t n_reads, uint32_t max_len1, uint32_t max_len2, uint64_t *d_taxon_out, uint32_t *d_best_out,
                        uint32_t *d_compact_out, void *cuda_stream);

/* Several GPUs in ONE process (the counterpart of the reference's `-z N` consumer threads, kaiju.cpp:250-257): contexts created on different
 * devices over the same index and parameters; the batch is cut into contiguous shards, one host thread drives each context, results land
 * in the caller's arrays in input order.  Per-taxon counts stay per context (sum them, or all-reduce kj_counts_device_ptr()). */
int kj_classify_multi(kj_ctx **ctxs, int n_ctx, const char *seq1, const uint64_t *off1, const char *seq2, const uint64_t *off2,
                      uint64_t n_reads, uint64_t *taxon_out, uint32_t *best_out);
int kj_device_count(void);                        /* number of usable CUDA devices (0 = none) */

/* Whole files (SURVEY.md 8f-1; replaces the reader loop of kaiju.cpp:288-394 and the output formatting of
 * ConsumerThread.cpp:724-739): FASTA or FASTQ, plain or gzip, in2 = second file of paired-end reads or NULL.  The text is
 * parsed on the device (line splitting, name trimming at " /\t\r", strip() of non-letters), classified, and the output
 * lines "C\t<name>\t<taxid>" / "U\t<name>\t0" (verbose: plus "\t<best>\t<id,id,...,>") are formatted on the device and
 * written to out_path (NULL or "" = stdout) in INPUT order.  FASTQ = 4-line records; empty lines before the first and between
 * records are skipped as the reference's reader does (kaiju.cpp:288-289, 341-348).  Errors mirror the
 * reference's messages (file type detection, differing read names, file 1 longer than file 2) as KJ_ERR_IO. */
int kj_classify_files(kj_ctx *ctx, const char *in1, const char *in2, const char *out_path, int verbose,
                      uint64_t *n_reads_out, uint64_t *n_classified_out);

/* --- per-taxon read counts (SURVEY.md 8f-3: what kaiju2table's first pass computes, src/kaiju2table.cpp:186-245) --- */
/* Every successful kj_classify / kj_classify_verbose / kj_classify_files call adds its reads to a dense count vector in HBM:
 * one slot per taxon known to the context (all ids of nodes.dmp ascending, then DB taxa missing from it) + a last slot for
 * unclassified reads.  After kj_classify_device() the caller adds explicitly (kj_counts_add_device) once the launch is known
 * to be good.  With several GPUs the vectors are summed with one all-reduce over kj_counts_device_ptr() (uint64[kj_counts_size()]). */
int kj_counts_reset(kj_ctx *ctx);
uint64_t kj_counts_size(const kj_ctx *ctx);
void *kj_counts_device_ptr(kj_ctx *ctx);
int kj_counts_add_device(kj_ctx *ctx, const uint64_t *d_taxon, uint64_t n_reads, void *cuda_stream);
int kj_counts_get(kj_ctx *ctx, uint64_t *taxon_ids_out /* [size] or NULL; last = 0 */, uint64_t *counts_out /* [size] */);

/* kaiju2table's report (src/kaiju2table.cpp:150-365: header row, one row per taxon of `rank` by descending read count, then the
 * Viruses / "cannot be assigned" / threshold / unclassified rows) written from per-taxon counts instead of the per-read output file.
 * kj_table_write is host-only (ids[i] = 0 marks the unclassified reads); kj_counts_table feeds it the context's count vector.
 * label = the "file" column; append != 0 adds the rows of another data set to an existing report (no second header). */
typedef struct {
    const char *rank;             /* -r: phylum, class, order, family, genus or species           */
    double min_percent;           /* -m (default 0)                                               */
    int32_t min_read_count;       /* -c (default 0); only one of -m / -c                          */
    int32_t expand_viruses;       /* -e                                                           */
    int32_t filter_unclassified;  /* -u                                                           */
    int32_t full_path;            /* -p                                                           */
    const char *rank_list;        /* -l: comma-separated ranks, or NULL                           */
} kj_table_opts;
int kj_table_write(const uint64_t *taxon_ids, const uint64_t *counts, uint64_t n, const char *nodes_dmp, const char *names_dmp,
                   const char *label, const kj_table_opts *opts, const char *out_path, int append);
int kj_counts_table(kj_ctx *ctx, const char *nodes_dmp, const char *names_dmp, const char *label, const kj_table_opts *opts,
                    const char *out_path, int append);

/* Per-read work queues on the device are sized from worst-case bounds; should one overflow anyway, the affected launch is
 * flagged (never silently truncated).  kj_classify() checks this itself; after kj_classify_device() call kj_check_errors()
 * once the stream has finished: KJ_OK, or KJ_ERR_OVERFLOW (the results of that launch are invalid).  When the overflow was
 * the Greedy substituted-variant ring (the reference's heap is unbounded; pathological -e/-s settings on long reads), the
 * library enlarges the ring, so repeating the call succeeds -- kj_classify() does that internally. */
int kj_check_errors(kj_ctx *ctx);

/* --- index construction: protein FASTA -> .fmi (what `kaiju-mkbwt -a ALPHABET -e E` followed by `kaiju-mkfmi` writes, byte for byte) --- */
/* The generalized suffix array (every sequence followed by its own terminator; terminators sort below all letters and among
 * themselves by input order), the BWT, the sampled suffix array and the compact FM index are all built on the device: prefix
 * doubling with hand-written radix sorts, re-sorting only the suffixes that are still tied.  The host parses the FASTA with
 * kaiju-mkbwt's rules (readFasta.c, sequence.c) and writes the files.  Limits: fewer than 2^32 rows (residues + sequences),
 * at most 24 letters.  A '*' (the terminator character) inside a sequence is refused: kaiju-mkbwt reads it as a sequence end
 * and writes a BWT shorter than its own header.  Bytes >= 0x80 are skipped like other non-letters. */
#define KJ_MKFMI_MAX_ROUNDS 40
typedef struct {
    int32_t chpt_exp;             /* -e: a suffix-array sample every 2^chpt_exp rows (0..16; kaiju-makedb uses 5, tests 3)      */
    const char *alphabet;         /* -a: the letters (NULL = "ACDEFGHIKLMNPQRSTVWY"), or "protein" (= the 20 residues + X)     */
    int32_t write_bwt_sa;         /* also write <prefix>.bwt and <prefix>.sa as kaiju-mkbwt does                              */
} kj_mkfmi_opts;
typedef struct {
    int64_t bwtlen;               /* rows: residues + sequences                                                                */
    int32_t nseq;
    int32_t sort_rounds;          /* radix-sorted rounds: the initial one on packed letters + the prefix-doubling ones        */
    uint64_t round_items[KJ_MKFMI_MAX_ROUNDS];   /* suffixes sorted in each round (round 0 = all of them)                   */
    uint64_t sort_bytes;          /* bytes the sort kernels read and write (keys, values, histograms), over all rounds        */
    double parse_ms, upload_ms, sort_ms, assemble_ms, write_ms;   /* wall time of the stages                                  */
} kj_mkfmi_stats;
/* KJ_ERR_UNSUPPORTED: >= 2^32 rows, more than 24 letters, no sequence in the input, '*' in a sequence; KJ_ERR_NOMEM: the device
 * memory estimate (about 45 bytes per row) exceeds the free memory; KJ_ERR_NO_DEVICE without a GPU.  stats may be NULL. */
int kj_mkfmi(const char *faa_path, const char *out_prefix, const kj_mkfmi_opts *opts, int device, kj_mkfmi_stats *stats);

/* --- introspection --- */
const char *kj_last_error(void);                  /* thread-local text of the last failure          */
uint64_t kj_kernel_launches(const kj_ctx *ctx);   /* number of kernels this context has launched    */
uint64_t kj_index_bytes(const kj_ctx *ctx);       /* bytes of HBM held by the index                 */
double kj_last_kernel_ms(const kj_ctx *ctx);      /* device time of the last classify kernel (CUDA events) */
int kj_launch_geometry(const kj_ctx *ctx, int *grid, int *block, int *dyn_smem_bytes);  /* of the last classify launch */
int kj_version(void);
/* test hooks: checksums of the index arrays (rank, letters, sa_tax, seq_tax, kmer | bwtlen, wide, n_sa) as held in HBM by a context,
 * and the same from the host transcoder (no GPU needed) -- the device construction is tested against the host one array for array */
int kj_debug_index_checksums(kj_ctx *ctx, uint64_t out[8]);
int kj_debug_host_index_checksums(const kj_index_view *index, const kj_taxonomy_view *taxonomy, uint64_t out[8]);

#ifdef __cplusplus
}
#endif
#endif
