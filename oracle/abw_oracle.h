/* TEST INFRASTRUCTURE ONLY -- flat-array CPU restatement of the abawaca hot path.
 *
 * This is the parity oracle for the CUDA path (tests/, __graft_entry__.smoke()
 * and bench.py's cpu_baseline leg are its only users; the product never calls
 * it).  Every function cites the reference lines it follows.  It is pinned
 * against the compiled reference itself (oracle/_ref, built from
 * /root/reference/src by oracle/Makefile) by tests/test_oracle_vs_reference.py
 * and the committed fixtures under tests/golden/.
 *
 * Conventions: scaffold and datapoint (dp) indices are 0-based here; the
 * reference's are 1-based (ScafDpData.cpp:90-101).  Dimension numbers in result
 * records are 1-based like the reference's (ClusterData.cpp:187).
 */
#ifndef ABW_ORACLE_H
#define ABW_ORACLE_H
#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ABWO_NKMER_DIMS 180   /* 2 + 10 + 32 + 136 canonical 1..4-mers, abawaca-build.cpp:75-100 */

typedef struct {
	uint32_t scaf;        /* 0-based scaffold index */
	uint32_t pos0;        /* 0-based leftmost reference position (ReadMapping.cpp:41) */
	uint32_t len;         /* read length = SEQ.size() (ReadMapping.h:44) */
	uint32_t flag_nsnps;  /* low 16 bits: SAM FLAG; high 16 bits: num_snps() */
} abwo_read;

typedef struct {
	uint32_t cluster_ndps_threshold;   /* 100, ClusterSeparator.h:72 */
	double   sensitivity_threshold;    /* 0.8, ...BySensitivitySpecificity.h:42 */
	double   specificity_threshold;    /* 0.8, :43 */
	double   product_threshold;        /* 0.8, :44 */
	double   sum_threshold;            /* 1.6, :45 */
	double   scg_overlap_threshold;    /* 0.2, ClusterQuality.cpp:130 */
	uint64_t scg_min_size;             /* 500000, ClusterQuality.cpp:119 */
	double   fraction_dps_in;          /* 0.8, ...SplitScafs.h:59 */
	double   split_scaf_ratio_threshold; /* 0.1, ...SplitScafs.h:44 */
	uint32_t max_snps;                 /* 15, abawaca-build.cpp:437 */
	uint32_t window_size;              /* 2000, abawaca-build.cpp:436 */
} abwo_params;

void abwo_default_params(abwo_params* p);

/* ---- feature stage -------------------------------------------------------------------------- */

/* String.cpp:37-51: upper-case in place; returns -1 if ok, else the index of a lower-case 'n' (which throws). */
int64_t abwo_validate_upper(char* seq, uint64_t len);
/* String.cpp:114-146 */
uint64_t abwo_count_N(const char* seq, uint64_t len);
double abwo_gc(const char* seq, uint64_t len);
/* abawaca-build.cpp:198-228.  1-based inclusive coordinates.  Returns the number of segments
 * (writes at most cap of them). */
uint64_t abwo_segment(const char* seq, uint64_t len, uint64_t window, uint64_t* seg_start, uint64_t* seg_end, uint64_t cap);
/* abawaca-build.cpp:75-100: name of each of the 180 dims in .lrn order ("A" first, not written to .lrn). */
const char* abwo_kmer_dim_name(int dim);
/* canonical dim of a k-mer given as 2-bit code (A=0,C=1,G=2,T=3, first base most significant) */
int abwo_kmer_dim_of(int k, uint32_t code);
/* abawaca-build.cpp:103-174: the 180 un-truncated frequencies of one segment. counts (optional, may be NULL):
 * raw window counts for k=1..4 laid out [4][16][64][256] = 340 entries, and totals[4]. */
void abwo_kmer_features(const char* seg, uint64_t len, double out[ABWO_NKMER_DIMS], uint32_t* counts340, uint32_t totals[4]);
/* abawaca-build.cpp:603: int(1000.0*x)/1000.0 */
double abwo_trunc3(double x);
/* abawaca-build.cpp:177-185,231-244,546-551: add the reads of ONE sample, in array order.
 * seg_first[s]..seg_first[s+1] index the segments of scaffold s.  cov is [nseg] for this sample.
 * scaf_nbps (may be NULL) accumulates read lengths per scaffold (the -c sample, :242-243). */
void abwo_coverage(const abwo_read* reads, uint64_t nreads, const uint64_t* seg_first, const uint64_t* seg_start, const uint64_t* seg_end,
                   uint32_t nscaf, uint32_t max_snps, double* cov, uint64_t* scaf_nbps);

/* Whole feature stage over a concatenated assembly (OpenMP over scaffolds).  First call with rows==NULL to
 * size: returns the number of segments.  rows is [nseg][179 + nsamples] holding the TRUNCATED values that
 * abawaca-build writes to .lrn (dim "A" dropped, abawaca-build.cpp:585-603); raw (may be NULL) is
 * [nseg][180 + nsamples] un-truncated.  seg_scaf/seg_start/seg_end describe every segment.
 * info_* (may be NULL): per scaffold length-normalised coverage of sample `this_sample` (trunc3), gc (trunc3), Ns. */
uint64_t abwo_build_features(const char* seq, const uint64_t* offsets, uint32_t nscaf, const abwo_params* p,
                             const abwo_read* const* reads, const uint64_t* nreads, uint32_t nsamples, int this_sample,
                             uint32_t* seg_scaf, uint64_t* seg_start, uint64_t* seg_end, uint64_t* seg_nonN,
                             double* rows, double* raw, double* info_cvg, double* info_gc, uint64_t* info_Ns);

/* ---- split search --------------------------------------------------------------------------- */

typedef struct {
	const double*   values;   /* column-major [D][N] */
	uint64_t        N;
	uint32_t        D;
	const uint32_t* dp2scaf;  /* [N] 0-based */
	uint32_t        S;
	const uint32_t* T;        /* [S] scaf_db.ndps(scaf): GLOBAL number of dps of the scaffold */
	const uint64_t* len;      /* [S] sequence length */
	const uint64_t* scgmask;  /* [S][W] */
	uint32_t        W;
} abwo_search_data;

typedef struct {
	int32_t  found;       /* 0: no candidate at all (best_separation untouched: dimension -1) */
	uint32_t dim;         /* 1-based */
	double   value;
	double   a;           /* sens/spec strategy: sensitivity;  split-scafs strategy: split_scaf_ratio */
	double   b;           /* sens/spec strategy: specificity;  split-scafs strategy: cluster_size_ratio */
	int32_t  legal;
} abwo_best;

enum { ABWO_SENS_SPEC = 0, ABWO_SPLIT_SCAFS = 1 };

/* ...Specificity.cpp:91-161 / ...SplitScafs.cpp:79-154 + ClusterSeparator.cpp:11-16 + ClusterQuality.cpp:96-136:
 * best separation of the cluster made of `dps` (n of them), over all dimensions. */
void abwo_separate(const abwo_search_data* d, const abwo_params* p, int strategy, const uint32_t* dps, uint64_t n, abwo_best* best);

/* ClusterSeparator.cpp:25-54,82-134: children of a legal best separation.  side[i] in {1,2} for dps[i] after
 * scaffold re-homing; raw_side[i] before re-homing (raw_dps_cluster1/2); assigned[s] in {0,1,2} per scaffold.
 * Returns 1 if both children have >= cluster_ndps_threshold dps (the split stands), 0 if rejected. */
int abwo_children(const abwo_search_data* d, const abwo_params* p, const uint32_t* dps, uint64_t n, uint32_t dim1, double value,
                  uint8_t* side, uint8_t* raw_side, uint8_t* assigned, uint64_t* n1, uint64_t* n2);

typedef struct {
	uint32_t id, parent;
	uint64_t ndps;
	uint32_t nscafs;          /* assigned scaffolds */
	int32_t  split;           /* 1: split into child1/child2; 0: terminal */
	abwo_best best;           /* as left in best_separation after separate() (reset when a legal split was rejected) */
	uint32_t child1, child2;
	uint64_t child1_ndps, child2_ndps;
	uint32_t child1_nscafs, child2_nscafs;
	uint64_t child1_raw, child2_raw;
	/* terminal clusters: ClusterQuality::total_size / scg (ClusterQuality.cpp:44-48,78-87; SCGdb.cpp:6-18,41-55) */
	uint64_t total_size;
	uint32_t scg_unique;
	double   scg_avg;
} abwo_cluster_rec;

/* abawaca.cpp:95-197: the breadth-first work list from the all-inclusive cluster 1.  recs has room for cap
 * records; returns the number of evaluated clusters.  dp2cluster [N] / scaf2cluster [S]: terminal cluster id, 0 if none. */
uint32_t abwo_run(const abwo_search_data* d, const abwo_params* p, int strategy, abwo_cluster_rec* recs, uint32_t cap,
                  uint32_t* dp2cluster, uint32_t* scaf2cluster, int nthreads);

/* SCGdb.cpp:6-18,41-55 over a scaffold list; a scaffold listed more than once counts once (the reference walks a std::set) */
void abwo_cluster_scg(const abwo_search_data* d, const uint32_t* scafs, uint32_t nscafs, uint32_t* nunique, double* avg);

#ifdef __cplusplus
}
#endif
#endif
