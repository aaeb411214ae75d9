/* xmapper_b200 — C ABI of the B200-native X-Mapper aligner stage.
 *
 * Drop-in boundary: replaces the body of mapper.AlignerWorker.process()/align() in mathjeff/Mapper @ ae7f346a
 * (src/main/java/mapper/AlignerWorker.java:157-261; constructor state :22-33) — a batch of queries in, the
 * List<QueryAlignments> the AlignmentListeners receive (:652-656) out.  Everything left of the boundary
 * (options, file writers) stays the host's: the reference's Java host, whose binding a maintainer adds (Panama FFM / JNI), is shown
 * in INTEGRATION.md; `python -m mapper_b200` is this project's own host.
 *
 * All pointers are HOST memory unless stated.  Every call returns 0 on success and a negative xm_status on
 * failure; xm_last_error(handle) returns the message (the host throws RuntimeException, matching
 * AlignerWorker.java:195-197).  There is no CPU fallback: without a CUDA device xm_create fails.
 *
 * Sequence layout (QV/SequenceBuilder.java:20-38, QV/Sequence.java:52-74): 4-bit IUPAC set codes
 * (A=1 C=2 G=4 T=8, N=15, QV/Basepairs.java), base i of a sequence at bits 4*(i&3) of 16-bit word i>>2.
 */
#ifndef XMAPPER_B200_H
#define XMAPPER_B200_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

typedef struct xm_handle xm_handle;
typedef struct xm_results xm_results;

enum xm_status {
  XM_OK = 0,
  XM_ERR_ARG = -1,          /* bad argument */
  XM_ERR_CUDA = -2,         /* no device / CUDA failure */
  XM_ERR_STATE = -3,        /* call order (reference or index missing) */
  XM_ERR_QUERY = -4         /* at least one query could not be aligned on the device; see xm_results q_status */
};

/* per-query status in xm_results (q_status) */
enum xm_query_status {
  XM_Q_OK = 0,
  XM_Q_AMBIGUOUS_QUERY = -2,  /* query with more than 64 IUPAC-ambiguous bases (MultiHashBlock conditions, HashBlock_ParentRow.java:97-120, are kept as 64-bit sets) */
  XM_Q_INDEX_TOO_SHORT = -3,  /* a seed needs a table longer than the index was built for (Readable_HashBlock_Database.java:108-113) */
  XM_Q_WORKSPACE = -5,        /* largest workspace tier exhausted */
  XM_Q_INTERNAL = -6          /* the reference would have thrown (e.g. PathAligner.java:159 on an empty queue) */
};

/* AlignmentParameters (src/main/java/mapper/AlignmentParameters.java:6-37) + HashBlock_Database options */
typedef struct xm_params {
  double mutation_penalty;            /* MutationPenalty */
  double insertion_start_penalty;     /* InsertionStart_Penalty */
  double insertion_extension_penalty; /* InsertionExtension_Penalty */
  double deletion_start_penalty;      /* DeletionStart_Penalty */
  double deletion_extension_penalty;  /* DeletionExtension_Penalty */
  double max_error_rate;              /* MaxErrorRate */
  double unaligned_penalty;           /* UnalignedPenalty */
  double ambiguity_penalty;           /* AmbiguityPenalty */
  double max_penalty_span;            /* Max_PenaltySpan */
  int32_t max_num_matches;            /* MaxNumMatches */
  int32_t enable_gapmers;             /* HashBlock_Database enableGapmers (Mapper.java:51) */
} xm_params;

/* new AlignerWorker(referenceProvider, parameters, duplicationDetector, ...) — AlignerWorker.java:22-33.
 * device: CUDA ordinal (one handle per GPU; one process per GPU in multi-GPU runs). */
int xm_create(const xm_params* params, int device, xm_handle** out);
void xm_destroy(xm_handle* h);
const char* xm_last_error(const xm_handle* h);

/* SequenceDatabase of the sorted reference (Mapper.sortAndComplementReference, Mapper.java:1151-1172; global
 * position space QV/SequenceDatabase.java:230-238): forward strands only, in database order; the reverse
 * complements are implicit (contig i occupies sequence ids 2i and 2i+1).
 * Global positions are as wide as the reference needs (QV/SequenceDatabase.java:69-74 sizes them by log2 of the forward + reverse
 * size; KAT T/PackedMap_Test.testLargeReferenceSize): 32 bits while 2 x total length <= 2^32, otherwise 40 bits, stored on the
 * device as a uint32 plane plus a uint8 plane so that the common case reads what it always read.  Limit: 2 x total < 2^40. */
int xm_set_reference(xm_handle* h, int32_t n_contigs, const uint16_t* const* packed4, const int32_t* lengths);

/* One PackedMap (PackedMap.java / QV/ByteKeyStore.java) per numBasepairsUsed, uploaded from the host's
 * HashBlock_Database: bucket b holds positions[offsets[b] .. offsets[b+1]) ascending global positions;
 * overfull[b] != 0 means "too many matches" (getNumMatchesLowerBound == Integer.MAX_VALUE).
 * capacity == 1 with no positions is the empty PackedMap(1, 1, ...) of HashBlock_Database.java:383-389. */
int xm_set_index_length(xm_handle* h, int32_t n_used, int32_t capacity, int32_t max_count, const int64_t* offsets,
                        const uint8_t* overfull, const uint32_t* positions);
/* The same call for references whose positions need more than 32 bits (required then; accepted for any reference). */
int xm_set_index_length_wide(xm_handle* h, int32_t n_used, int32_t capacity, int32_t max_count, const int64_t* offsets,
                             const uint8_t* overfull, const uint64_t* positions);
/* Declares HashBlock_Database.minInterestingSize (:51-55) and maxFullySetUpSize after all uploads. */
int xm_finish_index(xm_handle* h, int32_t min_interesting_size, int32_t max_built);

/* Alternative to the two calls above: build every table for numBasepairsUsed <= max_used from the uploaded
 * reference inside the library (HashBlock_Database.hashSequenceThroughSize/addHashblocks, :490-618).
 * n_threads == 0: built on the device (pyramid + gapmer kernel over reference slices, radix sorts, PackedMap fill kernel);
 * n_threads > 0: the library's host builder with that many threads (bit-identical tables; kept as the cross-check).
 * IUPAC-ambiguous ("-anc") references: both builders expand the reference's MultiHashBlocks (M/HashBlock_ParentRow.java:97-191)
 * and apply PackedMap.add(preventDuplicates) :117-131; the device builder gives every ambiguous 8 kbp slice a workspace of
 * XM_INDEX_AMB_ARENA_MB (default 64) MiB and returns XM_ERR_ARG, never a partial index, if an expansion outgrows it. */
int xm_build_index(xm_handle* h, int32_t max_used, int32_t n_threads);
/* Reads back a table (for parity tests against the host's PackedMaps). Pass NULL arrays to query sizes. */
int xm_get_index_length(xm_handle* h, int32_t n_used, int32_t* capacity, int32_t* max_count, int64_t* n_positions,
                        int64_t* offsets, uint8_t* overfull, uint32_t* positions);
int xm_get_index_length_wide(xm_handle* h, int32_t n_used, int32_t* capacity, int32_t* max_count, int64_t* n_positions,
                             int64_t* offsets, uint8_t* overfull, uint64_t* positions);
int xm_index_info(xm_handle* h, int32_t* min_interesting_size, int32_t* max_built);

/* Readable_DuplicationDetector table (Readable_DuplicationDetector.java:28-47): the sorted duplication start
 * keys of forward contig `contig`; window = DuplicationDetector.windowSize, granularity = getDetectionGranularity()
 * (DuplicationDetector.java:67-77). */
int xm_set_duplications(xm_handle* h, int32_t window, double granularity, int32_t contig, int32_t n, const int32_t* starts);
/* Or build it inside the library from the index (DuplicationDetector.process, :129-214; min_len / max_len < 0: the reference's
 * defaults, :59-65).  The bucket scan - lookupByForwardHash :41-52 for every bucket with >= min_copies positions, grouping by text -
 * runs on the device (xm_dup_scan_kernel, block lengths <= 64); saveDuplications' order-dependent containment rule (:332-436) is
 * applied to the blocks it finds on the host, in the reference's order. */
int xm_build_duplications(xm_handle* h, int32_t min_len, int32_t max_len, int32_t min_copies, int32_t window);
/* The same table computed entirely on host threads (any block length); kept as the cross-check of the device scan. */
int xm_build_duplications_host(xm_handle* h, int32_t min_len, int32_t max_len, int32_t min_copies, int32_t window);
int xm_get_duplications(xm_handle* h, int32_t contig, int32_t* n, int32_t* starts);

/* --infer-ancestors: AncestryDetector.unionRecentAncestors (M/AncestryDetector.java:89-147) over the handle's reference, set up as
 * M/Mapper.java:666-692 does it.  The handle's reference is replaced by the "-anc" reference: same contigs, same order, same lengths,
 * with IUPAC unions written where a recent common ancestor was inferred.  The index and the duplication table are discarded, as after
 * xm_set_reference (in every case: the call builds a temporary index of its own in their place).
 * min_interesting_size <= 0 / max_short_matches < 0: the HashBlock_Database defaults; Mapper passes (minDuplicationLength, 8) and
 * dissimilarity_threshold = MaxErrorRate / MutationPenalty.  *n_changed = forward positions whose code changed.
 * Runs on the device: index build, duplication-group scan (3 copies, window 1), the containment merge on the host, then one warp per
 * (group, direction) analysis and a kernel that writes the unions into the packed reference.  A position written twice
 * (OverriddenSequence.putEncoded) returns XM_ERR_STATE with "Cannot override contig <i>[-rev][<index>]: already overridden" (the
 * reference names the sequence instead of "contig <i>") and leaves the reference unchanged; so does every other error.
 * References with minDuplicationLength > 32 (over 2^32 bases) are not supported (XM_ERR_ARG). */
int xm_infer_ancestors(xm_handle* h, double dissimilarity_threshold, int32_t min_interesting_size, int32_t max_short_matches,
                       int32_t verify_no_duplicate_analyses, int64_t* n_changed);
/* Packed 4-bit codes of forward contig `contig` as the handle holds it now (ceil(length / 4) words; e.g. the "-anc" reference after
 * xm_infer_ancestors, for the host's own SequenceDatabase and writers). */
int xm_get_reference(xm_handle* h, int32_t contig, uint16_t* packed4);

/* AlignerWorker.process(): aligns n_queries queries. Query q owns n_seqs_per_query[q] (1 or 2) consecutive
 * sequences; sequence s is seq_len[s] bases at packed4 + seq_word_off[s] (16-bit words). seq_word_off holds
 * n_sequences + 1 entries: the last one is the total number of 16-bit words of packed4 (what gets copied to the device).
 * expected_inner / spacing_per_penalty are Query.expectedInnerDistance / spacingDeviationPerUnitPenalty
 * (QV/Query.java:17-30), ignored for single-sequence queries; NULL means 0.0 / 1.0 for every query.
 * *out is set to NULL first and only receives results when the call returns XM_OK or XM_ERR_QUERY (per-query failures,
 * see q_status); on every other error nothing is allocated for the caller to release. Blocking. */
int xm_align_batch(xm_handle* h, int32_t n_queries, const uint16_t* packed4, const int64_t* seq_word_off,
                   const int32_t* seq_len, const uint8_t* n_seqs_per_query, const double* expected_inner,
                   const double* spacing_per_penalty, xm_results** out);
/* Same, with every array already resident on the device of this handle (device pointers). Used by the
 * kernel-only timing leg of bench.py. */
int xm_align_batch_device(xm_handle* h, int32_t n_queries, const uint16_t* d_packed4, int64_t n_words,
                          const int64_t* d_seq_word_off, const int32_t* d_seq_len, const uint8_t* d_n_seqs_per_query,
                          const double* d_expected_inner, const double* d_spacing_per_penalty, int32_t max_seq_len,
                          xm_results** out);

/* Result = List<QueryAlignments> (QV/QueryAlignments.java:34-37) flattened CSR-style:
 *   query q           -> components  q_comp_off[q] .. q_comp_off[q+1]      (1, or 2 for unpaired mates)
 *   component c       -> choices     comp_choice_off[c] .. [c+1]           (QueryAlignment, QV/QueryAlignment.java:16-23)
 *   choice k          -> choice_f64[4k..] = spacingPenalty, overlapMultiplier, duplicationBonus, totalPenalty;
 *                        choice_inner[k] = totalDistanceBetweenComponents;
 *                        sequence alignments choice_sa_off[k] .. [k+1]
 *   seq alignment a   -> sa_contig[a] (forward contig index), sa_reversed[a] (referenceReversed),
 *                        sa_f64[2a..] = penalty, alignedPenalty (QV/SequenceAlignment.java:18-24);
 *                        blocks sa_block_off[a] .. [a+1]
 *   block b           -> blocks[4b..] = aStart, bStart, aLen, bLen (QV/AlignedBlock.java:6-19)
 * The arrays are assembled on the device and arrive in ONE transfer in a pinned host slab owned by the xm_results (the
 * pointers xm_results_array returns are views into it: a JNI/FFM host maps them as direct buffers); the slab goes back to a
 * small pool of the handle at xm_release_results.  Results of earlier batches stay valid while later batches run.
 */
enum xm_array {
  XM_Q_COMP_OFF = 0, XM_COMP_CHOICE_OFF = 1, XM_CHOICE_SA_OFF = 2, XM_SA_BLOCK_OFF = 3, /* int64 */
  XM_CHOICE_F64 = 4, XM_SA_F64 = 5,                                                     /* double */
  XM_CHOICE_INNER = 6, XM_SA_CONTIG = 7, XM_BLOCKS = 8, XM_Q_STATUS = 9,                /* int32 */
  XM_SA_REVERSED = 10,                                                                  /* uint8 */
  XM_STATS = 11,                                                                        /* int64: see xm_stat */
  XM_Q_CYCLES = 12                                                                      /* int64: per-query SM clock ticks, only when XM_QCYCLES=1 (profiling aid) */
};
enum xm_stat {
  XM_STAT_KERNEL_NS = 0,        /* device time of all kernels of this batch (CUDA events) */
  XM_STAT_LAUNCHES = 1,         /* launches of this library's own kernels (cub scans/sorts not counted) */
  XM_STAT_TIER0_QUERIES = 2, XM_STAT_TIER1_QUERIES = 3, XM_STAT_TIER2_QUERIES = 4,
  XM_STAT_PROBES = 5,           /* bucket-count probes (HashBlockPath.java:143-223) */
  XM_STAT_SEEDS = 6,            /* emitted seeds */
  XM_STAT_HITS = 7,             /* verified + rejected hits (Counting_HashBlockPath.java:93-153) */
  XM_STAT_STRAIGHT = 8,         /* StraightAligner calls */
  XM_STAT_PATH_CALLS = 9, XM_STAT_PATH_STEPS = 10, XM_STAT_PATH_CELLS = 11,
  XM_STAT_H2D_BYTES = 12, XM_STAT_D2H_BYTES = 13,
  XM_STAT_ALIGN_KERNEL_NS = 14, /* device time of the first-pass align kernel launch */
  XM_STAT_TIER0_NS = 15, XM_STAT_TIER1_NS = 16, XM_STAT_TIER2_NS = 17, /* device time of the align kernel per workspace tier */
  XM_STAT_CYC_SEED = 18, XM_STAT_CYC_STRAIGHT = 19, XM_STAT_CYC_HBA = 20, XM_STAT_CYC_PATH = 21, XM_STAT_CYC_TABLES = 22, XM_STAT_CYC_SPARE = 23,
  XM_STAT_CYC_TOTAL = 24,       /* SM clock ticks summed over queries, per phase (TOTAL only when XM_QCYCLES=1) */
  XM_STAT_EASY_QUERIES = 25, XM_STAT_EASY_NS = 26, /* first-pass kernel: queries in, device time */
  XM_STAT_EASY_DONE = 27,       /* queries the first-pass kernel completed */
  XM_STAT_EASY_PROBES = 28, XM_STAT_EASY_HITS = 29, XM_STAT_EASY_STRAIGHT = 30, /* counters of the queries completed by the first pass */
  XM_STAT_COUNT = 32
};
int64_t xm_results_array(const xm_results* r, int which, const void** ptr);
void xm_release_results(xm_results* r);

/* SAM bodies of the batch `r` came from, formatted on the device from its result arrays and the packed reads of the batch
 * (replaces QV/SamWriter.java:118-352 formatQueryAlignments/formatQueryAlignment/getSamFlags/getMappingQuality/formatNumber:
 * one line per sequence alignment, in query order; header lines and the file writer stay with the host).
 * Must be called before the next xm_align_batch on the handle (the device copy of the results is reused by it).
 * seq_names: the names of all sequences of the batch back to back (Sequence.getSourceName()), seq_name_off[n_sequences + 1];
 * contig_names / contig_name_off[n_contigs + 1]: Sequence.getName() of the contigs in xm_set_reference order.
 * *text stays valid until xm_release_results(r) or the next xm_format_sam on r. */
int xm_format_sam(xm_handle* h, xm_results* r, const char* seq_names, const int64_t* seq_name_off, const char* contig_names, const int64_t* contig_name_off,
                  const char** text, int64_t* n_bytes);

/* Count accumulation for --out-vcf/--out-mutations (replaces the MatchDatabase listener: QV/MatchDatabase.java:16-59,
 * QV/Alignments.java:89-156, QV/DirectionalAlignments.java:20-96).  xm_counts_enable allocates the state on the device; every
 * later xm_align_batch accumulates into it:
 *   - dense planes: reference-base depth in int32 units of 1/100 per [region: 0 middle, 1 end][direction: 0 forward, 1 reverse][position]
 *     (DirectionalAlignments.referenceCounts), read with xm_counts_fetch / xm_counts_device_ptr;
 *   - a sparse table of variants (alternates, deletions, insertion columns: DirectionalAlignments.alternates), read with
 *     xm_variants_fetch: entry i has
 *       keys[i]     = (global forward position) << 21 | region << 20 | direction << 19 | (insertion column + 1) << 3 | allele
 *                     global forward position = (sum of the lengths of the contigs before it) + position; insertion column + 1 == 0:
 *                     an allele AT the position (substitution or deletion), k + 1: column k of the insertion after the position;
 *                     allele = index into "ACGTN-" (AlignmentPosition_DirectionCounts.makeKeys)
 *       counts[i]   = Variant.count (sum of (int)(weight * 100))
 *       ex_gid[i]   = example read (Variant.exampleSequence): global sequence id << 1 | 1 if it is the "-rev" view
 *       ex_index[i] = Variant.exampleIndex (negative: deletion)
 *     entries are sorted by key; the example is the one DirectionalAlignments.betterExample (:63-96) would have kept.
 * xm_counts_batch_info (optional, before an xm_align_batch): the global id of the first sequence of the next batch (default: the
 * sequences are numbered in the order the handle receives them; a host that shards reads over GPUs passes the real ids) and, per
 * sequence, a key that orders the sequences like their names (Sequence.getName().compareTo, e.g. the rank of the name among the
 * names of the run; NULL: equal names assumed, ties fall to the id as in :92-95). */
int xm_counts_enable(xm_handle* h, double query_end_fraction);
int xm_counts_batch_info(xm_handle* h, int64_t first_sequence_id, const int64_t* seq_order_key, int64_t n_sequences);
int xm_counts_device_ptr(xm_handle* h, void** d_ptr, int64_t* n_int32);
int xm_counts_fetch(xm_handle* h, int32_t contig, int32_t* out /* 4 * contig length */);
int xm_variants_fetch(xm_handle* h, int64_t* n, uint64_t* keys, int32_t* counts, int64_t* ex_gid, int32_t* ex_index /* NULL arrays: size query */);

/* VCF and mutations BODIES formatted on the device from the count planes and the variant table (QV/VcfFormatterWorker.java:27-159,
 * QV/MutationsFormatterWorker.java:25-147 over QV/FilteredAlignments; the headers embed the command line and stay with the host, as
 * do the file writer and the order of the contigs: VcfWriter / MutationsWriter visit them in the TreeMap order of their names,
 * :111-114, and the library does not sort names).  The host asks for one forward contig and a range of positions [start, end) at a
 * time, of any size it likes:
 *   - the VCF text of any split of [0, contig length) concatenates to the text of the whole contig;
 *   - so does the mutations text of any split at multiples of 8192 (start % 8192 == 0, end % 8192 == 0 or end == contig length):
 *     a run of deletions is reported per writer job of 8192 positions, so a run that crosses a job boundary is two records.
 * The text is placed in a pinned host buffer owned by the handle; *text stays valid until the next xm_format_vcf /
 * xm_format_mutations on the handle, or xm_destroy.  Format calls are ordered with xm_align_batch on the same handle.  Every
 * entry point of this library may be called by concurrent threads on one handle.
 * After xm_counts_reduce every rank holds the planes and the table of the whole run, so any rank can format any contig and the
 * ranks may split the contigs between them.
 * Errors: counts not enabled -> XM_ERR_STATE; a bad contig or range, a mutations range not on the 8192 grid -> XM_ERR_ARG. */
/* MutationDetectionParameters (QV/MutationDetectionParameters.java): the six thresholds of FilteredAlignments.  All zero (or a NULL
 * filter) = MutationDetectionParameters.emptyFilter(). */
typedef struct xm_variant_filter {
  float min_snp_total_depth, min_snp_depth_fraction;
  float min_indel_start_total_depth, min_indel_start_depth_fraction;
  float min_indel_continuation_total_depth, min_indel_continuation_depth_fraction;
} xm_variant_filter;
/* The reads the VCF support column can show: the distinct global sequence ids (ascending) of the examples of the current variant
 * table.  gids == NULL: size query.  Reduces pending records first, like xm_variants_fetch. */
int xm_variants_examples(xm_handle* h, int64_t* n, int64_t* gids);
/* The forward texts of exactly those sequences, in that order: gids as xm_variants_examples listed them, then the reads packed as
 * xm_align_batch takes them (seq_word_off has n + 1 entries).  The "-rev" view of an example (ex_gid & 1) is made on the device.
 * A count, id or order that differs from xm_variants_examples, or a read whose length is not the length of the read that was
 * counted, returns XM_ERR_ARG.  The upload belongs to the table as it is now: a later batch, xm_counts_reduce or xm_counts_enable
 * makes it stale. */
int xm_variants_set_examples(xm_handle* h, int64_t n, const int64_t* gids, const uint16_t* packed4, const int64_t* seq_word_off, const int32_t* seq_len);
/* VcfFormatterWorker.format over positions [start, end) of forward contig `contig`, named contig_name: body lines only.
 * show_support != 0 needs the examples of the current table (xm_variants_set_examples), else XM_ERR_STATE; show_support == 0 needs
 * none.  Reference characters are the handle's reference codes (IUPAC letters on ambiguous references). */
int xm_format_vcf(xm_handle* h, int32_t contig, const char* contig_name, int64_t start, int64_t end, const xm_variant_filter* f,
                  int32_t include_non_mutations, int32_t show_support, const char** text, int64_t* n_bytes);
/* MutationsFormatterWorker.format over [start, end) of forward contig `contig` (start % 8192 == 0; end % 8192 == 0 or end == contig
 * length); needs no examples. */
int xm_format_mutations(xm_handle* h, int32_t contig, const char* contig_name, int64_t start, int64_t end, const xm_variant_filter* f,
                        const char** text, int64_t* n_bytes);

/* Read ingestion (the FASTA/FASTQ readers and M/SequenceSplitter.java:9-38 in front of Mapper.compare): text in, the arrays
 * xm_align_batch takes out.  Parses the complete records at the start of text[0, n_bytes).
 *   - Records.  FASTA: a '>' header line followed by any number of sequence lines up to the next '>' (any line width; blank lines are
 *     skipped).  FASTQ: exactly four lines, "@name", the sequence, '+' with anything after it, and a quality line as long as the
 *     sequence (multi-line FASTQ is not supported).  "\r\n" line ends are accepted.
 *   - Bases.  The 15 IUPAC letters of QV/Basepairs, in either case, become their 4-bit codes.  Any other byte in a sequence line, a
 *     quality line of the wrong length, a missing '+' line, a FASTQ record not starting with '@', text before the first FASTA header or
 *     a FASTQ input ending inside a record returns XM_ERR_ARG; xm_last_error names the record (index within this call) and the byte offset.
 *   - Names.  The header line after its marker, to the end of the line, without a trailing '\r' (the reference's FastaParser was not
 *     available to check this choice against).
 *   - Chunking.  A record is complete when its last line ends in '\n', or when at_eof != 0; a FASTA record only once the next header
 *     is seen (or at_eof).  *n_consumed = the bytes of the complete records parsed (all n_bytes when at_eof and every record was taken);
 *     the caller passes the rest again, followed by the next chunk.  At most max_records records are parsed (< 0: no limit): a
 *     paired-end caller takes the same number of records from both files.
 *   - Splitting.  split_size > 0: a record longer than split_size becomes n = (len - 1) / split_size + 1 sequences, piece k covering
 *     [len*k/n, len*(k+1)/n) and named "name[start:end]" (SURVEY.md §5; unchecked against the reference's splitter).  XM_R_RECORD maps
 *     every sequence back to its record.
 * The text goes to the device through a pinned staging buffer; line ends (one ballot per warp over the bytes, then a scan), record
 * bounds, lengths, the split, word offsets, packing, names and the checks run there (kernels xm_parse_*, on a stream of their own, so a
 * call overlaps an xm_align_batch on the same handle); the arrays come back in one copy into a pinned slab owned by the xm_reads.
 * n_bytes < 2^31 per call. */
enum xm_text_format { XM_FASTA = 0, XM_FASTQ = 1 };
typedef struct xm_reads xm_reads;
int xm_parse_reads(xm_handle* h, int32_t format, const char* text, int64_t n_bytes, int32_t at_eof,
                   int64_t max_records, int32_t split_size, xm_reads** out, int64_t* n_consumed);
enum xm_reads_array {
  XM_R_PACKED = 0,        /* uint16: packed4, the layout xm_align_batch takes */
  XM_R_SEQ_WORD_OFF = 1,  /* int64, n + 1 */
  XM_R_SEQ_LEN = 2,       /* int32 */
  XM_R_NAME_OFF = 3,      /* int64, n + 1, into XM_R_NAMES */
  XM_R_NAMES = 4,         /* char */
  XM_R_RECORD = 5         /* int64: index within this call of the record a sequence came from */
};
/* Element count of array `which` of r (n = number of sequences), *ptr = its first element; valid until xm_release_reads(r). */
int64_t xm_reads_array(const xm_reads* r, int which, const void** ptr);
void xm_release_reads(xm_reads* r);

/* Measurement aid (bench.py's roofline): sustained issue rates of this GPU, in warp-instructions per second over the whole chip,
 * from three micro-benchmark kernels timed with CUDA events - out[0] INT32 (IMAD chains), out[1] FP64 (DADD chains), out[2] FP32
 * FFMA chains (full-rate pipe: the issue-slot ceiling); out[3] = number of SMs, out[4] = maximum SM clock in Hz.  SURVEY.md §8(d) takes the relevant
 * peaks of this path (instruction issue, FP64 pipe) from such a measurement on the box rather than from a datasheet. */
int xm_measure_peaks(xm_handle* h, double* out /* 5 doubles */);

/* Multi-GPU reduction of the count planes inside the library (NCCL over NVLink; libnccl.so.2 is loaded at run time).
 * One process (or thread) per GPU, as the reference runs one AlignerWorker per thread and MatchDatabase merges them
 * (QV/MatchDatabase.java:16-59): rank 0 calls xm_comm_unique_id and hands the 128 bytes to the others by any means,
 * every rank calls xm_comm_init on its handle (collective), and xm_counts_reduce (collective, blocking) leaves the int32 sum over
 * all ranks in every rank's planes (ncclAllReduce: exact and order-free) and the union of all ranks' variant tables, reduced by
 * key, in every rank's table (sizes all-gathered, entries exchanged with grouped ncclBroadcast, device sort + reduce-by-key).
 * Call it once, after the last batch: a second call would add the already-summed planes again. */
int xm_comm_unique_id(uint8_t* id128);
int xm_comm_init(xm_handle* h, int32_t n_ranks, int32_t rank, const uint8_t* id128);
int xm_counts_reduce(xm_handle* h);
/* Measurement aid: of the latest xm_counts_reduce, the device time of the ncclAllReduce of the planes (CUDA events) and the time the
 * exchange + merge of the variant table took after it. */
int xm_counts_reduce_times(xm_handle* h, double* planes_allreduce_ms, double* variants_ms);

#ifdef __cplusplus
}
#endif
#endif
