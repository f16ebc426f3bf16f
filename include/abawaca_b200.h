/* abawaca_b200 -- C ABI of the B200-native abawaca hot path.
 *
 * The reference (CK7/abawaca) has no FFI layer; its seams are C++ constructors and virtuals
 * (SURVEY.md section 8b).  This header is what a maintainer of the reference binds instead of
 * those seams; INTEGRATION.md shows the C++ adapter for each.  Every entry point
 *   - is extern "C", takes plain pointers and sizes, returns an int status (0 = ok),
 *   - never throws and never takes ownership of caller memory,
 *   - is callable from one host thread per context; abw_last_error(ctx) holds the text.
 * Pointers named h_* are host memory, d_* device memory; plain names follow the `on_device` flag.
 *
 * Index conventions: scaffolds and datapoints (dps) are 0-based here (the reference's are 1-based,
 * ScafDpData.cpp:90-101); scaffolds must be in byte-wise name order and dps grouped by scaffold in
 * dp-name order, which is what abawaca-build writes and ScafDpData builds.  Dimension numbers in
 * result records are 1-based like the reference's (ClusterData.cpp:187).
 */
#ifndef ABAWACA_B200_H
#define ABAWACA_B200_H
#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ABW_OK                 0
#define ABW_ERR_CUDA           1
#define ABW_ERR_ARG            2
#define ABW_ERR_ILLEGAL_DNA    3   /* lower-case 'n': the reference throws Illegal_DNAString (String.cpp:47-49) */
#define ABW_ERR_UNSUPPORTED    4
#define ABW_ERR_NOMEM          5

#define ABW_NKMER_DIMS 180         /* canonical 1..4-mers, abawaca-build.cpp:75-100 */

typedef struct abw_ctx abw_ctx;
typedef struct abw_seqset abw_seqset;     /* packed assembly on the device */
typedef struct abw_segments abw_segments; /* the datapoints (windows) of an assembly */
typedef struct abw_search abw_search;     /* one split-search problem resident on the device */

/* Constants compiled into the reference's hot path (SURVEY.md section 5), as a POD. */
typedef struct {
	uint32_t cluster_ndps_threshold;     /* 100     ClusterSeparator.h:72 */
	double   sensitivity_threshold;      /* 0.8     ClusterSeparatorBySensitivitySpecificity.h:42 */
	double   specificity_threshold;      /* 0.8     :43 */
	double   product_threshold;          /* 0.8     :44 */
	double   sum_threshold;              /* 1.6     :45 */
	double   scg_overlap_threshold;      /* 0.2     ClusterQuality.cpp:130 */
	uint64_t scg_min_size;               /* 500000  ClusterQuality.cpp:119 */
	double   fraction_dps_in;            /* 0.8     ClusterSeparatorSplitScafs.h:59 */
	double   split_scaf_ratio_threshold; /* 0.1     ClusterSeparatorSplitScafs.h:44 */
	uint32_t max_snps;                   /* 15      abawaca-build.cpp:437 */
	uint32_t window_size;                /* 2000    abawaca-build.cpp:436 */
	/* Not in the reference: candidates scoring below min(min_reported_score, product_threshold) are not
	 * examined.  That cannot change any split (a best separation below product_threshold fails is_legal,
	 * whatever the other thresholds are), but the best separation reported for a TERMINAL cluster is
	 * then only found if it scores at least that much.  Set to 0 to also reproduce the reference's log
	 * line for terminal clusters. */
	double   min_reported_score;
} abw_params;

typedef struct {
	uint32_t scaf;        /* 0-based scaffold index; >= nscaf: reference name not in the assembly (skipped, abawaca-build.cpp:549-550) */
	uint32_t pos0;        /* 0-based leftmost reference position = SAM POS - 1 (ReadMapping.cpp:41) */
	uint32_t len;         /* read length = SEQ.size() (ReadMapping.h:44) */
	uint32_t flag_nsnps;  /* low 16 bits: SAM FLAG; high 16 bits: num_snps() from MD:Z/CIGAR (ReadMapping.cpp:78-185) */
} abw_read;

/* ---- context -------------------------------------------------------------------------------- */
int         abw_ctx_create(int device, abw_ctx** out);
void        abw_ctx_destroy(abw_ctx* ctx);
const char* abw_last_error(const abw_ctx* ctx);
const char* abw_version(void);
void        abw_default_params(abw_params* p);
/* number of kernel launches issued through this context so far (bench.py reports it) */
uint64_t    abw_kernel_launches(const abw_ctx* ctx);
/* number of device blocks this context had to obtain from the driver so far (0 per pass once its block cache is warm) */
uint64_t    abw_arena_misses(const abw_ctx* ctx);
/* Debug allocator (environment ABW_REDZONE=1, or =abort): every device block of the library is surrounded by canary zones, handed out filled with 0xFF,
   never reused, and verified when it is released; this is the number of blocks found damaged so far in this process (always 0 when the mode is off).
   It stands in for compute-sanitizer memcheck where that tool cannot be run (DESIGN.md section 9). */
uint64_t    abw_redzone_violations(void);
/* the stream every kernel of this context is launched on (a cudaStream_t), for event timing */
void*       abw_ctx_stream(const abw_ctx* ctx);
int         abw_ctx_synchronize(abw_ctx* ctx);
/* Per-kernel device timing for profiling runs: while enabled every launch is bracketed by CUDA events on the context
 * stream and waited for (so launches are serialised; do not enable it in a timed region).  abw_profile_report writes
 * "kernel<TAB>launches<TAB>total_ms" lines into buf and returns the size needed. */
int         abw_profile_enable(abw_ctx* ctx, int on);
size_t      abw_profile_report(abw_ctx* ctx, char* buf, size_t cap);

/* ---- feature stage (abawaca-build) ------------------------------------------------------------ */

/* Replaces Bio::DNAString construction for every scaffold read by SeqIORead_fasta<DNASequence>::next_seq
 * (SeqIORead_fasta.h:51-103, String.cpp:37-51): upper-cases, keeps A/C/G/T as 2-bit codes, marks every
 * other character in a validity mask and the literal 'N' in a second mask (quirk Q2).
 * ascii: concatenated scaffold sequences; offsets[nscaf+1] (host) delimit them. */
int abw_pack_sequences(abw_ctx* ctx, const char* ascii, int ascii_on_device, const uint64_t* h_offsets, uint32_t nscaf, abw_seqset** out);
void abw_seqset_destroy(abw_seqset* s);
/* Bio::Ns and the C+G count behind Bio::gc, per scaffold (String.cpp:114-146); host arrays [nscaf] */
int abw_seqset_stats(abw_ctx* ctx, const abw_seqset* s, uint64_t* h_count_N, uint64_t* h_count_GC);

/* Replaces Scaf::Scaf (abawaca-build.cpp:198-228): cuts every scaffold into windows of equal non-N length. */
int abw_segment(abw_ctx* ctx, const abw_seqset* s, uint32_t window_size, abw_segments** out);
void abw_segments_destroy(abw_segments* g);
uint64_t abw_segments_count(const abw_segments* g);
/* host copies (any pointer may be NULL): seg_first[nscaf+1], and per segment scaffold, 1-based inclusive start/end, non-N bases */
int abw_segments_get(abw_ctx* ctx, const abw_segments* g, uint64_t* h_seg_first, uint32_t* h_seg_scaf, uint64_t* h_seg_start, uint64_t* h_seg_end, uint64_t* h_seg_nonN);

/* the same per-window arrays into PINNED host buffers on the copy stream (like abw_d2h_async: overlaps what is enqueued next, complete after
 * abw_ctx_synchronize); the segments object must stay alive until then */
int abw_segments_get_async(abw_ctx* ctx, const abw_segments* g, uint32_t* h_seg_scaf, uint64_t* h_seg_start, uint64_t* h_seg_end, uint64_t* h_seg_nonN);

#define ABW_FEAT_TRUNC3 0   /* int(1000*x)/1000.0, the value abawaca-build prints with %.3lf (abawaca-build.cpp:603) */
#define ABW_FEAT_RAW    1   /* the un-truncated double */
/* Replaces Scaf_segment::Scaf_segment (abawaca-build.cpp:103-174).  Writes, for every segment, the 180 canonical
 * k-mer frequencies into columns [col0, col0+180) of the row-major matrix `rows` (row stride ld doubles).
 * With skip_A != 0 the first dimension ("A", which abawaca-build does not write, :585-602) is dropped and 179 columns are written. */
int abw_kmer_features(abw_ctx* ctx, const abw_seqset* s, const abw_segments* g, int kind, int skip_A, double* d_rows, uint64_t ld, uint32_t col0);

/* Replaces the SAM loop body abawaca-build.cpp:546-551 with Scaf::add_mapped_read (:231-244) and
 * Scaf_segment::add_mapped_read (:177-185) for ONE sample: reads in SAM order.  Writes column `col` of `rows`.
 * d_scaf_nbps (may be NULL): per scaffold sum of accepted read lengths (the -c sample, :242-243), uint64 [nscaf].
 * With reads_on_device != 0 the call returns once the work is enqueued on the context stream (like every entry point, later calls on the
 * same context see its results; a host that reads d_rows through its own stream calls abw_ctx_synchronize first). */
int abw_coverage(abw_ctx* ctx, const abw_segments* g, const abw_read* reads, uint64_t nreads, int reads_on_device, uint32_t max_snps,
                 int kind, double* d_rows, uint64_t ld, uint32_t col, uint64_t* d_scaf_nbps);

/* Several samples in one call, in any of the record formats.  ABW_READS_FULL: abw_read records, the read filter (:546-550) is applied on the device.
 * ABW_READS_COMPACT: abw_read8 records of the reads that PASSED that filter on the host (SURVEY.md section 8b(4): the host parser may pre-filter), in SAM
 * order, 8 bytes instead of 16 over the host link; every read is `len` bases long unless len16 gives per-read lengths (reads longer than 65535 bases
 * need the full format).  Record arrays (and len16) are DEVICE memory; h2d_ticket (0: none) is the abw_h2d_async ticket they depend on -- the call
 * waits for it on the device just before the sample's first kernel, so the records of later samples may still be in flight when it is made.
 * Writes columns [col0, col0 + nsamples) of `rows`.  With three-decimal output the windows whose third decimal depends on the order of the reads
 * (DESIGN.md section 4) are collected over ALL samples and go through one stable sort instead of one per sample.
 * this_sample (-1: none): index of the -c sample whose accepted read lengths are added to d_scaf_nbps (:242-243). */
typedef struct {
	uint32_t scaf;        /* 0-based scaffold index */
	uint32_t pos0;        /* SAM POS - 1 */
} abw_read8;
#define ABW_READS_FULL    0
#define ABW_READS_COMPACT 1
/* ABW_READS_SORTED: the reads of ABW_READS_COMPACT (host-filtered, in SAM order) in about 2 bytes per read when the SAM file is coordinate sorted.
 * The reads are cut into runs of one scaffold each, runs[nruns]: `count` consecutive reads on scaffold `scaf` (a scaffold may appear in several runs,
 * in any order; a count may be 0).  `reads` points to uint16_t delta[nreads]: read i's pos0 is prev + delta[i], prev being the pos0 of read i - 1 when
 * that read is in the same run and 0 for the first read of a run.  delta 0xFFFF is an escape: pos0 is then exc[k], k = number of escapes before read i
 * (an encoder escapes every difference that is negative or >= 0xFFFF).  Lengths as in the compact format (len, or len16).  Nothing is reordered, so
 * the result is that of the compact records of the same reads.  The arrays may still be in flight behind h2d_ticket, so malformed contents are dealt
 * with on the device: reads past the sum of the counts, reads of runs with scaf >= nscaf and escapes with k >= nexc are skipped (an escaped read that
 * is skipped counts as pos0 0 for the read after it); counts past nreads are ignored.  Decoded into 8-byte records in device memory of the context
 * that live until the call returns. */
#define ABW_READS_SORTED  2
typedef struct {
	uint32_t scaf;        /* 0-based scaffold index */
	uint32_t count;       /* consecutive reads on it */
} abw_read_run;
typedef struct {
	const void*     reads;       /* abw_read[nreads], abw_read8[nreads] or uint16_t delta[nreads], device memory */
	uint64_t        nreads;
	int32_t         format;
	uint32_t        len;         /* compact, sorted: read length when len16 is NULL */
	const uint16_t* len16;       /* compact, sorted, optional: per-read lengths, device memory */
	uint64_t        h2d_ticket;
	/* sorted only (zero for the other formats): device memory, nruns < 2^32, nexc <= nreads */
	const abw_read_run* runs;
	uint64_t        nruns;
	const uint32_t* exc;         /* escaped positions in read order */
	uint64_t        nexc;
} abw_sample;
int abw_coverage_batch(abw_ctx* ctx, const abw_segments* g, const abw_sample* h_samples, uint32_t nsamples, uint32_t max_snps, int kind, double* d_rows, uint64_t ld,
                       uint32_t col0, int32_t this_sample, uint64_t* d_scaf_nbps);

/* The values abawaca-build prints are multiples of 0.001 (int(1000*x)/1000.0, abawaca-build.cpp:603): columns [col0, col0 + ncols) of the row-major
 * matrix as integer thousandths, row-major [nrows][ncols] of uint16_t (bits = 16; k-mer frequencies are at most 1000) or uint32_t (bits = 32; coverage),
 * a quarter / half of the bytes for the trip to the host; k / 1000.0 gives back the identical double.  Enqueued on the context stream; *d_inexact
 * (device int32, set to 0 by the caller) is incremented for every value that is not exactly k / 1000.0 with k in range -- the caller then fetches the doubles. */
int abw_rows_to_milli(abw_ctx* ctx, const double* d_rows, uint64_t nrows, uint64_t ld, uint32_t col0, uint32_t ncols, int bits, void* d_out, int32_t* d_inexact);

/* ---- SAM text -> read records on the device (SURVEY.md section 8f row 1) ------------------------------------------------
 * abw_names: the scaffold names as a device-side hash table; name i is names_blob[h_name_off[i] .. h_name_off[i+1]) and gets index i
 * (replaces the std::map<string, Scaf*> lookup scafs.find(ref_name), abawaca-build.cpp:482,549). */
typedef struct abw_names abw_names;
int  abw_names_create(abw_ctx* ctx, const char* names_blob, const uint64_t* h_name_off, uint32_t nscaf, abw_names** out);
void abw_names_destroy(abw_names* n);
/* Replaces SAMReader::next_mapping (ReadMappingReader.cpp:80-116), ReadMapping::ReadMapping(const char*) (ReadMapping.cpp:23-72) and the SNP count
 * of ReadMapping::determine_snps (ReadMapping.cpp:78-185) for one chunk of SAM text that ends at a line boundary (the caller carries an
 * unfinished last line over to the next chunk).  Every line that is neither empty nor a '@' header line becomes one abw_read, in file
 * order, written to d_reads[0 .. *nreads) (device memory, capacity cap records): scaf = index of RNAME (0xFFFFFFFF if unknown),
 * pos0 = POS - 1, len = length of SEQ, flag_nsnps = FLAG | num_snps << 16.  If the chunk holds more than cap records nothing is written,
 * *nreads holds the number needed and ABW_ERR_ARG is returned.  Errors the reference throws on are reported as a status:
 * lower-case 'n' in SEQ (ABW_ERR_ILLEGAL_DNA), fewer than 11 fields or a malformed MD:Z description (ABW_ERR_ARG). */
int abw_parse_sam(abw_ctx* ctx, const abw_names* names, const char* text, uint64_t nbytes, int text_on_device, abw_read* d_reads, uint64_t cap, uint64_t* nreads);

/* ---- FASTA text -> packed assembly on the device -----------------------------------------------------------------------
 * Replaces SeqIORead_fasta<DNASequence>::next_seq (SeqIORead_fasta.h:51-103, with SeqIORead::getline(true), SeqIORead.h:85-121) for a whole
 * file: lines are trimmed of white space on both ends, blank lines skipped, a line starting with '>' opens a record whose id is the text up
 * to the first white space, every other line is appended to the open record (interior white space included).
 * abw_fasta_scan indexes the text (kept on the device; a device text must stay alive until abw_fasta_destroy) and returns ABW_ERR_ARG where
 * the reference throws Bad_file (sequence text before the first header, '>' followed by white space).  abw_fasta_get returns, per record in
 * file order, where its id lies in the text and how long its sequence is; the host reads the names from its own copy of the text, decides
 * the order (abawaca-build keeps the first record of every name, in name order: std::map::insert, abawaca-build.cpp:482-490) and
 * abw_fasta_pack builds the abw_seqset of records h_order[0 .. nout) exactly as abw_pack_sequences would from the concatenated sequences. */
typedef struct abw_fasta abw_fasta;
int      abw_fasta_scan(abw_ctx* ctx, const char* text, uint64_t nbytes, int text_on_device, abw_fasta** out);
void     abw_fasta_destroy(abw_fasta* f);
uint64_t abw_fasta_count(const abw_fasta* f);
int      abw_fasta_get(abw_ctx* ctx, const abw_fasta* f, uint64_t* h_id_off, uint32_t* h_id_len, uint64_t* h_seq_len);
int      abw_fasta_pack(abw_ctx* ctx, const abw_fasta* f, const uint32_t* h_order, uint32_t nout, abw_seqset** out);

/* ---- assembly in 2 bits per base -> packed assembly on the device ----------------------------------------------------------
 * The codes are those of a UCSC .2bit file: T=0 C=1 A=2 G=3, four bases per byte, the first base in the HIGH bits of its byte; every scaffold
 * starts at a byte of its own (at any byte address).  Characters other than A/C/G/T (either case) are described by runs: kind ABW_BASE_N for the
 * literal 'N', ABW_BASE_OTHER for any other character (quirk Q2: a base for windowing that breaks k-mers); the code under a run is ignored.
 * abw_pack_2bit builds the abw_seqset abw_pack_sequences makes from the ASCII text the encoding stands for, bit for bit (packed, valid, nmask,
 * Bio::Ns and the C+G count).  Upper/lower case is not part of the encoding, so a lower-case 'n' cannot be reported here: encoders refuse it.
 * Checked on the host (ABW_ERR_ARG): h_byte_off[s] + ceil(h_len[s] / 4) <= nbytes and h_len[s] < 2^32.  The runs may still be in flight behind
 * h2d_ticket, so their contents are dealt with on the device: a run with scaf >= nscaf or start >= the scaffold's length is skipped, a run that
 * reaches past the scaffold's end is clipped, a position under any N run is N whatever other runs cover it, and a kind other than ABW_BASE_N
 * counts as ABW_BASE_OTHER.  The call waits for h2d_ticket on the device and returns once its work is enqueued; codes and runs must stay alive
 * until later work on the context has consumed the result (e.g. until abw_ctx_synchronize). */
#define ABW_BASE_N     0   /* the literal 'N': nmask bit set, valid bit clear */
#define ABW_BASE_OTHER 1   /* any other non-ACGT character: valid bit clear */
typedef struct {
	uint32_t scaf;        /* 0-based scaffold index */
	uint32_t start;       /* 0-based first position in the scaffold */
	uint32_t len;         /* positions */
	uint32_t kind;        /* ABW_BASE_N or ABW_BASE_OTHER */
} abw_base_run;
typedef struct {
	const uint8_t*      codes;        /* device: 2-bit codes in the UCSC .2bit layout */
	uint64_t            nbytes;       /* readable bytes at codes */
	const uint64_t*     h_byte_off;   /* host [nscaf]: byte of codes where scaffold s starts */
	const uint64_t*     h_len;        /* host [nscaf]: bases of scaffold s, < 2^32 */
	const abw_base_run* runs;         /* device [nruns], may be NULL when nruns is 0 */
	uint64_t            nruns;
	uint64_t            h2d_ticket;   /* 0: none; codes and runs may still be in flight behind it (abw_h2d_async) */
} abw_2bit_assembly;
int abw_pack_2bit(abw_ctx* ctx, const abw_2bit_assembly* in, uint32_t nscaf, abw_seqset** out);

/* UCSC .2bit files, the counterpart of abw_fasta_*.  abw_twobit_scan parses header, index and record headers of the file image h_file[nbytes] on the
 * host: versions 0 (32-bit offsets) and 1 (64-bit offsets), either byte order (the signature 0x1A412743 read byte-swapped marks a big-endian file).
 * ABW_ERR_ARG for a malformed file: truncated, an offset or block outside the file or the sequence, blocks unsorted or overlapping, an empty name.
 * abw_twobit_get returns per record, in file order, where its name lies in the file, the name's length and the sequence length.
 * abw_twobit_decode writes record `record` as twoBitToFa prints its sequence: upper case, lower case under mask blocks, 'N' (or 'n' under a mask
 * block) under N blocks; h_out has room for the sequence length.
 * abw_twobit_pack packs the records h_order[0 .. nout) (abawaca-build keeps the first record of every name, in name order) from d_file, the same
 * file image in device memory (possibly still in flight behind h2d_ticket), through abw_pack_2bit.  ABW_ERR_ILLEGAL_DNA when a selected record has
 * an N block that overlaps a mask block: that is a lower-case 'n' in its FASTA, which the reference throws on (String.cpp:47-49). */
typedef struct abw_twobit abw_twobit;
int      abw_twobit_scan(abw_ctx* ctx, const void* h_file, uint64_t nbytes, abw_twobit** out);
void     abw_twobit_destroy(abw_twobit* t);
uint64_t abw_twobit_count(const abw_twobit* t);
int      abw_twobit_get(abw_ctx* ctx, const abw_twobit* t, uint64_t* h_name_off, uint32_t* h_name_len, uint64_t* h_seq_len);
int      abw_twobit_decode(abw_ctx* ctx, const abw_twobit* t, uint64_t record, const void* h_file, char* h_out);
int      abw_twobit_pack(abw_ctx* ctx, const abw_twobit* t, const void* d_file, uint64_t h2d_ticket, const uint32_t* h_order, uint32_t nout, abw_seqset** out);

/* ---- .lrn data lines -> matrix on the device ---------------------------------------------------------------------------------
 * Replaces the datapoint loop of ClusterData::ClusterData (ClusterData.cpp:110-168) for the text after the four header lines: every line that is
 * not empty and does not start with '%' is "<key>\t<v1>\t...\t<vD>"; keys are read with atoi, values with atof (:151,159).  Row r of the
 * file goes to d_keys[r] and d_values[r*D .. r*D+D) (device memory, room for cap_rows rows); *nrows = rows found.  The matrix can be handed to
 * abw_search_create as it is (ABW_LAYOUT_ROWMAJOR, values_on_device, h_row_of_dp built from the keys).  Decimal values take the exact
 * one-operation conversion on the device; the rare others (more than 19 digits, exponents beyond +-22, inf/nan) are converted with the host's atof. */
int abw_parse_lrn(abw_ctx* ctx, const char* text, uint64_t nbytes, int text_on_device, uint32_t D, uint64_t* d_keys, double* d_values, uint64_t cap_rows, uint64_t* nrows);
/* Row i of d_dst (row stride ld_dst) = the first ncols values of row rows[i] of d_src (row stride ld_src), for i < nrows; both matrices row-major
 * doubles in device memory, rows in host memory (rows_on_device = 0) or device memory.  E.g. the rows abw_parse_lrn read, in file order, put
 * into datapoint order.  Enqueued on the context stream. */
int abw_gather_rows(abw_ctx* ctx, const double* d_src, uint64_t ld_src, const uint64_t* rows, int rows_on_device, uint64_t nrows, uint32_t ncols, double* d_dst,
                    uint64_t ld_dst);

/* ---- matrix -> .lrn data lines on the device (the counterpart of abw_parse_lrn) ---------------------------------------------------------------
 * Replaces the per-value printf of the .lrn writers: abawaca-build's abawaca.lrn ("\t%.3lf", abawaca-build.cpp:603) and ClusterEsomWriter's
 * clusters/<id>.lrn ("\t%lf", ClusterWriter.cpp:81-98).  Line i (line0 <= i < nlines) is "<r+1>\t<v_0>\t...\t<v_{ncols-1}>\n" with r = rows[i]
 * (rows == NULL: r = i) and v_c = d_values[r * ld + col0 + c] (row-major doubles, device memory); rows is device memory when rows_on_device != 0.
 * Every value is byte-identical to what the C library's printf writes for the format: ties round to even, the sign of zero is kept, inf / nan
 * are "inf", "-inf", "nan", "-nan".  The longest run of whole lines from line0 on that fits `cap` bytes is written to d_text (device memory);
 * *nlines_done / *nbytes say how many lines and bytes that is, and the caller continues with line0 + *nlines_done.  If line line0 alone does not
 * fit, nothing is written, *nbytes holds its size and ABW_ERR_ARG is returned.  d_text may start at any byte address.  Values of magnitude >= 2^64 / 10^decimals and non-finite values
 * are printed by the host's C library; all others on the device. */
#define ABW_TEXT_3LF 0   /* "%.3lf": abawaca.lrn */
#define ABW_TEXT_LF  1   /* "%lf":   clusters/<id>.lrn */
int abw_format_lrn(abw_ctx* ctx, const double* d_values, uint64_t ld, uint32_t col0, uint32_t ncols, const uint64_t* rows, int rows_on_device,
                   uint64_t line0, uint64_t nlines, int fmt, char* d_text, uint64_t cap, uint64_t* nlines_done, uint64_t* nbytes);

/* device memory helpers so that hosts without a CUDA runtime binding can drive the ABI */
int abw_device_alloc(abw_ctx* ctx, size_t bytes, void** d_out);
int abw_device_free(abw_ctx* ctx, void* d_ptr);
int abw_copy_to_device(abw_ctx* ctx, void* d_dst, const void* h_src, size_t bytes);
int abw_copy_to_host(abw_ctx* ctx, void* h_dst, const void* d_src, size_t bytes);
int abw_memset_device(abw_ctx* ctx, void* d_ptr, int byte, size_t bytes);
/* Staging that overlaps compute: abw_h2d_async enqueues a copy from PINNED host memory on the context's copy stream and
 * returns a ticket; abw_wait_h2d makes every later call on this context wait (on the device, not the host) for that copy.
 * Typical use: enqueue the assembly and all samples' read records up front, then wait for each just before its
 * abw_pack_sequences / abw_coverage call.  Tickets are retired by abw_ctx_synchronize. */
int abw_h2d_async(abw_ctx* ctx, void* d_dst, const void* h_src, size_t bytes, uint64_t* ticket);
int abw_wait_h2d(abw_ctx* ctx, uint64_t ticket);
/* Device-to-host copy into PINNED host memory on the copy stream, ordered after everything enqueued on the context so far and overlapping
 * whatever is enqueued next (e.g. the .lrn matrix travels back while the split search runs).  Complete after abw_ctx_synchronize. */
int abw_d2h_async(abw_ctx* ctx, void* h_dst, const void* d_src, size_t bytes);

/* ---- split search (abawaca) ----------------------------------------------------------------- */

#define ABW_SENS_SPEC   0   /* ClusterSeparatorBySensitivitySpecificity (live, abawaca.cpp:109) */
#define ABW_SPLIT_SCAFS 1   /* ClusterSeparatorSplitScafs (compiled, not instantiated, abawaca.cpp:110) */

#define ABW_LAYOUT_COLMAJOR 0  /* values[d * ld + dp] */
#define ABW_LAYOUT_ROWMAJOR 1  /* values[dp * ld + d] (the .lrn layout written by abw_kmer_features/abw_coverage) */
#define ABW_LAYOUT_ROWMAJOR_MILLI32 2  /* `values` points to uint32_t k[dp * ld + d] in DEVICE memory, the value being (double)k / 1000.0: what abw_rows_to_milli
                                          (bits = 32) writes.  Every .lrn value is int(1000 x) / 1000.0 (abawaca-build.cpp:603), so nothing is lost; half the bytes
                                          when ranks exchange feature columns (the dimension-sharded search of bench.py at N > 1) */

/* Replaces ClusterData(lrn, scaf_db) + ScafDpData + SCGdb as the split search sees them (ClusterData.cpp:27,
 * ScafDpData.cpp:91-99, SCGdb.cpp:86-117): N datapoints x D dimensions, dp2scaf[N] (non-decreasing),
 * T[S] = scaf_db.ndps(scaf) (must be >= 2: ScafDpData drops scaffolds with one dp, quirk Q1),
 * len[S] = sequence length, scgmask[S][W] = bit set of SCG names per scaffold.
 * h_dp2scaf may be NULL when the matrix holds all T datapoints of every scaffold in scaffold order (N = sum of T, the reference's own flow).
 * The value matrix has nrows rows; datapoint i is row h_row_of_dp[i] of it (NULL: nrows = N and datapoint i is row i).
 * This is how the rows of scaffolds with a single window, which abawaca-build writes but ScafDpData drops, are skipped
 * without copying the matrix.  The all-inclusive cluster 1 (init_cluster, abawaca.cpp:242-251) is the root.
 * A matrix in device memory (values_on_device) is read where it lies, also by abw_search_run (the separating value of a split is looked up in it):
 * it must stay valid and unchanged until the search object is destroyed.  A host matrix is copied to the device once, in its own layout. */
int abw_search_create(abw_ctx* ctx, const double* values, int values_on_device, int layout, uint64_t ld, uint64_t nrows, const uint64_t* h_row_of_dp,
                      uint64_t N, uint32_t D, const uint32_t* h_dp2scaf, uint32_t S, const uint32_t* h_T, const uint64_t* h_len, const uint64_t* h_scgmask, uint32_t W,
                      const abw_params* params, int strategy, abw_search** out);
/* The same for the matrix of a feature build that is still on the device (abw_kmer_features / abw_coverage* wrote d_rows, one row per window of g):
 * T = windows per scaffold, scaffolds with fewer than two windows are dropped as ScafDpData does (ScafDpData.cpp:92-93), the datapoints are the rows of
 * the kept scaffolds -- all derived on the device, no trip through the host.  h_len / h_scgmask are indexed by the scaffolds of the ASSEMBLY [nscaf].
 * *S_out / *N_out: kept scaffolds and their datapoints; h_kept[0 .. *S_out) (room for nscaf entries, may be NULL): the assembly index of every kept
 * scaffold, i.e. what scaffold i of the search results refers to. */
int abw_search_create_from_features(abw_ctx* ctx, const abw_segments* g, const double* d_rows, uint64_t ld, uint32_t D, const uint64_t* h_len, const uint64_t* h_scgmask,
                                    uint32_t W, const abw_params* params, int strategy, uint32_t* S_out, uint64_t* N_out, uint32_t* h_kept, abw_search** out);
void abw_search_destroy(abw_search* s);

typedef struct {
	int32_t  found;     /* 0: best_separation untouched (dimension -1, ClusterSeparator.h:21) */
	uint32_t dim;       /* 1-based */
	double   value;
	double   a;         /* sensitivity            | split_scaf_ratio   */
	double   b;         /* specificity            | cluster_size_ratio */
	int32_t  legal;     /* ClusteringResult::is_legal */
} abw_best;

typedef struct {
	uint32_t id, parent;
	uint64_t ndps;
	uint32_t nscafs;            /* assigned scaffolds */
	int32_t  split;             /* ClusterSeparator::separate() returned true */
	abw_best best;              /* best_separation after separate() (reset when the children were too small, ClusterSeparator.cpp:125-132) */
	uint32_t child1, child2;    /* ids handed out at split time, cluster1 first (abawaca.cpp:164-193) */
	uint64_t child1_ndps, child2_ndps;
	uint32_t child1_nscafs, child2_nscafs;
	uint64_t child1_raw, child2_raw;   /* |raw_dps_cluster1/2| before scaffold re-homing */
	uint64_t total_size;        /* terminal clusters: ClusterQuality::total_size */
	uint32_t scg_unique;        /* terminal clusters: SCGdb::num_unique_scgs */
	double   scg_avg;           /* terminal clusters: SCGdb::average_num_copies_for_unique_scgs */
	/* terminal clusters, when abw_search_set_scaffold_stats was called (else -1): ClusterQuality::gc / cvg (ClusterQuality.cpp:51-75),
	 * length-weighted mean and standard deviation over the assigned scaffolds in scaffold order (standard_deviation, :6-27) */
	double   gc_avg, gc_sd, cvg_avg, cvg_sd;
} abw_cluster_rec;

/* Replaces the work-list loop abawaca.cpp:98-197 with ClusterSeparator::separate() (ClusterSeparator.cpp:57-135) inside:
 * evaluates clusters breadth first (= ascending id), level by level, until every cluster is terminal.
 * h_recs[cap] receives one record per evaluated cluster in id order; *nrecs the number evaluated.
 * h_dp2cluster[N] / h_scaf2cluster[S] (may be NULL): terminal cluster id, 0 if none (abawaca.cpp:199-210). */
int abw_search_run(abw_ctx* ctx, abw_search* s, abw_cluster_rec* h_recs, uint32_t cap, uint32_t* nrecs, uint32_t* h_dp2cluster, uint32_t* h_scaf2cluster);

/* ---- dimension-sharded search over several GPUs (one process per GPU) ---------------------------------------------------
 * Every rank holds ALL datapoints but only a contiguous block of dimensions (abw_search_create on that block, then
 * abw_search_set_shard).  Per level each rank sweeps its dimensions; the per-cluster best records are all-gathered and
 * merged with the reference's total order (ClusterSeparator.cpp:11-16), the rank owning the winning dimension votes the
 * scaffolds (ClusterSeparator.cpp:94-101) and the result reaches the others through a sum in which every other rank
 * contributes zeros.  The two collectives are supplied by the caller (NCCL through torch.distributed in bench.py; any MPI
 * would do): they act on DEVICE buffers of this rank and must have completed when they return. */
typedef struct {
	int (*allgather)(void* user, const void* d_send, void* d_recv, size_t bytes_per_rank);   /* recv = rank 0 | rank 1 | ... */
	int (*allreduce_sum_i64)(void* user, void* d_buf, size_t count);                         /* in place, 64-bit integer sum */
	void* user;
	int rank, world;
	/* non-zero: the operations are enqueued on the context stream (abw_ctx_stream) and complete in its order, so a whole search is enqueued without a
	 * host wait (abw_nccl_collectives_create).  Zero: they are host synchronous -- the library waits for its stream before every call and the
	 * operation has completed when the callback returns. */
	int stream_ordered;
} abw_collectives;
int abw_search_set_shard(abw_search* s, uint32_t dim_offset, uint32_t D_total);
/* The same with interleaved dimensions: this rank holds the dimensions dim_offset + k * dim_stride (k = 0 .. D-1) of D_total, in that order in its matrix.
 * Round-robin shards (dim_offset = rank, dim_stride = world) give every rank the same mix of k-mer and coverage dimensions (SURVEY.md section 8e). */
int abw_search_set_shard_strided(abw_search* s, uint32_t dim_offset, uint32_t dim_stride, uint32_t D_total);
int abw_search_run_sharded(abw_ctx* ctx, abw_search* s, const abw_collectives* coll, abw_cluster_rec* h_recs, uint32_t cap, uint32_t* nrecs,
                           uint32_t* h_dp2cluster, uint32_t* h_scaf2cluster);

/* Native collectives: NCCL operations enqueued on the context stream (no host synchronisation).  libnccl.so.2 is resolved at run time
 * (ABW_ERR_UNSUPPORTED if it cannot be found; set ABW_NCCL_LIB to its path).  Rank 0 obtains an id and hands its ABW_NCCL_ID_BYTES bytes to
 * the other ranks by any means; every rank then creates its abw_collectives, on its own context. */
#define ABW_NCCL_ID_BYTES 128
int  abw_nccl_unique_id(abw_ctx* ctx, void* id128);
int  abw_nccl_collectives_create(abw_ctx* ctx, const void* id128, int rank, int world, abw_collectives* out);
void abw_nccl_collectives_destroy(abw_collectives* c);

/* ---- column exchange between the ranks over NVLink peer memory (CUDA IPC; one process per GPU on one node) --------------------------------
 * Between the scaffold-sharded feature build and the dimension-sharded search every rank needs its columns (rank, rank + world, ...) of
 * everybody's rows.  Each rank allocates one exchange buffer and exports it; abw_peer_group_create maps the buffers of all ranks; then
 * abw_scatter_columns_milli reads the local rows once and stores, for every rank q, the integer thousandths (see abw_rows_to_milli) of q's columns
 * straight into q's buffer: q's matrix is uint32 [total rows][cnt(q)] at byte offset buf_offset_bytes of its buffer, cnt(q) = number of columns
 * c < ncols with c % world == q, and this rank's rows start at row row0 of it (row0 = rows of the ranks before it).  With `segs` (the windows the
 * rows belong to, one row per window) the rows of scaffolds with a single window are left out, as ScafDpData drops them (ScafDpData.cpp:92-93) and as
 * abw_search_create_from_features does; row0 then counts kept rows; NULL: every row is sent.  Conversion, column split and
 * transfer are one kernel on the context stream.  The receiver may read its buffer (abw_search_create, ABW_LAYOUT_ROWMAJOR_MILLI32, ld = cnt(q)) once
 * every rank's kernel has completed: order it with any stream-ordered collective of all ranks (a one-word abw_collectives.allreduce_sum_i64 will do),
 * and alternate between two halves of the buffer so that a rank that is a step ahead does not overwrite what a slower one still reads.
 * *d_inexact (device int32, may be NULL) is incremented when a value is not an exact multiple of 0.001 in [0, 2^31 / 1000).
 * ABW_ERR_UNSUPPORTED when CUDA IPC is not available (the caller then exchanges the columns with its own all-to-all). */
#define ABW_IPC_HANDLE_BYTES 64
typedef struct abw_peer_group abw_peer_group;
int  abw_peer_buffer_create(abw_ctx* ctx, size_t bytes, void** d_buf, unsigned char* handle64);
int  abw_peer_buffer_destroy(abw_ctx* ctx, void* d_buf);
int  abw_peer_group_create(abw_ctx* ctx, void* d_own, const unsigned char* handles /* [world][ABW_IPC_HANDLE_BYTES], entry `rank` is ignored */, int rank, int world,
                           abw_peer_group** out);
void abw_peer_group_destroy(abw_peer_group* g);
int  abw_scatter_columns_milli(abw_ctx* ctx, const abw_peer_group* g, const abw_segments* segs, const double* d_rows, uint64_t nrows, uint64_t ld, uint32_t ncols,
                               uint64_t row0, size_t buf_offset_bytes, int32_t* d_inexact);

/* Per-scaffold G+C fraction and coverage (ScafDpData::Seq::get_gc / get_cvg, the .info columns), host arrays [S]: the terminal records then
 * carry the summary.txt statistics ClusterQuality::gc and ClusterQuality::cvg compute.  Call between abw_search_create and abw_search_run. */
int abw_search_set_scaffold_stats(abw_ctx* ctx, abw_search* s, const double* h_gc, const double* h_cvg);

/* Stop after `max_levels` levels of the breadth-first search (0 = run to the end).  With 1 this is exactly one
 * ClusterSeparator::separate() call on the root: record 0 describes the split and dp2cluster/scaf2cluster hold the ids of
 * the two children (2 = cluster1, 3 = cluster2), which is what a per-cluster adapter needs (INTEGRATION.md section 1). */
int abw_search_set_max_levels(abw_search* s, uint32_t max_levels);

/* Counters of the last abw_search_run, and -- only while abw_profile_enable(ctx, 1) is in force, because measuring them makes the host wait
 * for the device several times per level -- milliseconds of device time per kernel family (CUDA events on the context stream), else 0 */
typedef struct {
	float build_ms;       /* abw_search_create: key transform, sort, element packing */
	float sweep_ms;       /* threshold-sweep kernels, all levels */
	float partition_ms;   /* stable partition kernels, all levels */
	float other_ms;       /* reductions, children, SCG tables */
	uint64_t sweep_elements;     /* sum over levels of (dps x dimensions) swept */
	uint64_t partition_elements;
	uint32_t levels;
	uint32_t sweep_launches;
} abw_search_profile;
int abw_search_get_profile(const abw_search* s, abw_search_profile* out);

/* ClusterQuality::scg (ClusterQuality.cpp:44-48) for an arbitrary scaffold list: the number of distinct SCG names on the scaffolds (nunique) and
 * the average number of copies per distinct name (avg, 0 when there is none).  The list is taken as a set, as the reference's std::set is: a
 * scaffold listed more than once counts once.  An index >= the number of scaffolds of the search gives ABW_ERR_ARG. */
int abw_cluster_scg(abw_ctx* ctx, const abw_search* s, const uint32_t* h_scafs, uint32_t nscafs, uint32_t* nunique, double* avg);

#ifdef __cplusplus
}
#endif
#endif
