// Split search of abawaca on the device (ClusterSeparator*.cpp, ClusterQuality.cpp, SCGdb.cpp).
//
// B200-first formulation (DESIGN.md section 3):
//   * every Dimension is sorted ONCE (abw_search_create).  A cluster only ever contains whole scaffold groups
//     (ClusterSeparator.cpp:104-122 re-homes datapoints to their scaffold's cluster), so the rank of a datapoint
//     inside its scaffold is a per-(datapoint, dimension) constant and the reference's incremental TP/FP counters
//     (ClusterSeparatorBySensitivitySpecificity.cpp:6-76) become prefix sums of per-element constants.
//   * per dimension the device keeps one u32 per datapoint, "element" = scaffold id | class | flags, ordered by value
//     and grouped by live cluster.  A level of the breadth-first search is
//        sweep      : stream the elements of every live (cluster, dimension) once, block scans, score candidates
//        reduce     : best candidate per cluster (score, then lowest dimension, then lowest value)
//        children   : scaffold majority vote + re-homing (ClusterSeparator.cpp:82-134)
//        partition  : stable 2-way partition of every dimension's element array by the scaffold's new cluster
//     instead of re-sorting every cluster (std::sort at ...Specificity.cpp:114) and rebuilding std::map/std::set state.
//   * the SCG acceptance test (ClusterQuality.cpp:96-136) is evaluated for EVERY candidate through a small per
//     (cluster, dimension) table indexed by the number of SCG-carrying scaffolds already flipped to side 1.
#include "features.cuh"
#include <algorithm>
#include <cmath>
#include <cstring>
#include <chrono>
#include <cstdlib>

namespace {

constexpr int      SW_THREADS = 256;
constexpr int      SW_ITEMS = 32;     // consecutive elements per thread: one 128-byte line, four 16-byte loads in flight
constexpr int      SW_TILE = SW_THREADS * SW_ITEMS;
constexpr uint32_t EL_SCAF_BITS = 27;
constexpr uint32_t EL_SCAF_MASK = (1u << EL_SCAF_BITS) - 1u;
constexpr uint32_t EL_CLASS_SHIFT = 27;     // 2 bits: sens/spec: 0 before the flip, 1 the flip element, 2 after
                                            //         split-scafs: position relative to r1 (0 below, 1 equal, 2 above)
constexpr uint32_t EL_AUX_SHIFT = 29;       // 2 bits: sens/spec: bit0 = flip element of an SCG-carrying scaffold
                                            //         split-scafs: position relative to r2
constexpr uint32_t EL_BOUNDARY = 1u << 31;  // value differs from the previous element of the same cluster
constexpr uint32_t EL_FLIP_BIT = 1u << EL_CLASS_SHIFT;        // classes are 0, 1, 2: the low class bit is set exactly for class 1 ...
constexpr uint32_t EL_CLS2_BIT = 2u << EL_CLASS_SHIFT;        // ... and the high one exactly for class 2

struct __align__(16) ScafRow { uint32_t T, n; uint64_t len; };

struct ClusterDesc {
	uint64_t off;        // first element of the cluster in every dimension's array
	uint32_t n;          // datapoints
	uint32_t kOff, K;    // segment of the per-dimension SCG scaffold list
	uint32_t tabOff;     // offset of the (K+1)-entry pass table (per dimension)
	uint32_t sOff, ns;   // segment of the scaffold list
	uint32_t totT;       // sum of T over the scaffolds of the cluster
	uint32_t U;          // number of scaffolds
	uint64_t totLen;     // sum of sequence lengths
	uint32_t ss_ok;      // split-scafs: every scaffold starts "in" cluster 2 (ClusterSeparatorSplitScafs.cpp:102-106)
	uint32_t tile0;      // first entry of the cluster in the level's tile table
	uint32_t fOff, nf;   // sens/spec: segment of the per-dimension flip list (scaffolds that can flip, in flip order)
};

struct CandRec {
	double   k1, k2;     // sens/spec: k1 = sens*spec (maximise).  split-scafs: k1 = ratio, k2 = size ratio (minimise)
	uint32_t p;          // number of datapoints with value <= candidate value
	uint32_t i0, i1, i2; // sens/spec: TP, total, TP+FP of the small side.  split-scafs: separated, in_small, in_large
	uint32_t found;
	uint32_t dim0;       // 0-based dimension (filled by the reduction; global index over all ranks of a sharded search)
};

constexpr uint32_t SCG_WMAX = 8;   // up to 512 distinct SCG names

// A live cluster of the current level, as the device keeps it (the work list of abawaca.cpp:98-197 lives on the device: no level waits for the host)
struct LevelCluster {
	ClusterDesc d;
	uint32_t id, parent, nassigned, pad;
	unsigned long long never[SCG_WMAX];      // SCG names on scaffolds that can never flip to side 1 of a sweep (n < T/2+1): always counted on side 2
};

// Control block of the breadth-first search, device resident.  The single-CTA kernels k_level_jobs / k_level_decide write it, every other kernel of a level
// reads its work sizes from it, so the host can enqueue level after level without knowing how many clusters, tiles or splits a level has.
struct LevelCtl {
	uint32_t C, TT, FPT, tab_total;          // current level: clusters, sweep tile-table entries, flip-prefix tile-table entries, pass-table entries per dimension
	uint32_t J, JM, CL_items, SS_items;      // best separations found, those whose dimension this rank holds, work items of k_count_low / k_scaf_sides
	uint32_t P, Tn, TM_items, term_blocks_done;   // splits, terminal clusters, work items of k_finalize_terminal, its CTAs that have finished
	uint32_t part_TT[4], part_tab_off[4], part_job_off[4];   // partition plans (scaffold list, elements, flip lists, SCG lists): tile-table entries and offsets
	unsigned long long part_item_end[4];      // cumulative work items of the plans (item = (dimension, tile-table entry))
	uint32_t next_id, nrec, level, done;
	uint32_t error, sweep_launches, ticks, done_at;   // ticks: levels executed, empty ones included; done_at: value of ticks after the level that ended the search
	unsigned long long tickets[4];            // flip-prefix, sweep, partition
	unsigned long long sweep_elements, partition_elements;
};

// what the host polls (mapped pinned memory): written by k_level_decide at the end of every level
struct LevelProgress {
	volatile uint32_t levels_done, done, error;
	volatile uint32_t ticks, done_at;                 // see LevelCtl; done_at is written before ticks
	volatile uint32_t c_next[16];                     // c_next[t & 15]: clusters of the level that follows the t-th executed level (t = 0, 1, ...)
};

template <int STRATEGY>
__device__ __forceinline__ bool cand_better(const CandRec& x, const CandRec& y)
{
	if(!x.found) return false;
	if(!y.found) return true;
	if(STRATEGY == ABW_SENS_SPEC) {
		if(x.k1 != y.k1) return x.k1 > y.k1;        // ...Specificity.h:28 (scores are never NaN here)
	}
	else {
		if(x.k1 != y.k1) return x.k1 < y.k1;        // ...SplitScafs.h:34-35
		if(x.k2 != y.k2) return x.k2 < y.k2;
	}
	if(x.dim0 != y.dim0) return x.dim0 < y.dim0;    // ClusterSeparator.cpp:13-14
	return x.p < y.p;                               // lower value <=> fewer datapoints at or below it (:15)
}

struct Agg {
	uint32_t a, b, c, d;
	unsigned long long e;
};
__device__ __forceinline__ Agg agg_zero() { Agg r; r.a = r.b = r.c = r.d = 0; r.e = 0; return r; }
__device__ __forceinline__ Agg agg_add(const Agg& x, const Agg& y)
{
	Agg r; r.a = x.a + y.a; r.b = x.b + y.b; r.c = x.c + y.c; r.d = x.d + y.d; r.e = x.e + y.e; return r;
}
__device__ __forceinline__ Agg agg_shfl_up(const Agg& x, int o)
{
	Agg r;
	r.a = __shfl_up_sync(0xffffffffu, x.a, o); r.b = __shfl_up_sync(0xffffffffu, x.b, o);
	r.c = __shfl_up_sync(0xffffffffu, x.c, o); r.d = __shfl_up_sync(0xffffffffu, x.d, o);
	r.e = __shfl_up_sync(0xffffffffu, x.e, o);
	return r;
}

// exclusive block scan of one Agg per thread, plus the block total.  smem: Agg[SW_THREADS/32 + 1]
__device__ __forceinline__ Agg block_excl_scan_agg(const Agg& v, Agg& total, Agg* sm)
{
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	Agg incl = v;
#pragma unroll
	for(int o = 1; o < 32; o <<= 1) {
		Agg t = agg_shfl_up(incl, o);
		if(lane >= o)
			incl = agg_add(incl, t);
	}
	if(lane == 31)
		sm[warp] = incl;
	__syncthreads();
	if(threadIdx.x == 0) {
		Agg run = agg_zero();
		for(int w = 0; w < SW_THREADS / 32; w++) {
			Agg t = sm[w];
			sm[w] = run;
			run = agg_add(run, t);
		}
		sm[SW_THREADS / 32] = run;
	}
	__syncthreads();
	Agg warp_ex = sm[warp];
	total = sm[SW_THREADS / 32];
	Agg ex = agg_add(warp_ex, incl);
	ex.a -= v.a; ex.b -= v.b; ex.c -= v.c; ex.d -= v.d; ex.e -= v.e;
	__syncthreads();
	return ex;
}

struct SweepParams {
	uint32_t thr;            // cluster_ndps_threshold
	double   min_score;      // min_reported_score
	float    prune;          // safe single-precision lower bound of min_score
	unsigned long long scg_min_size;
	double   fraction_in;    // split-scafs
};

// ---------------------------------------------------------------------------------------------------
// the threshold sweep: one CTA per tile of SW_TILE consecutive elements of a (cluster, dimension) segment.
// Work items are (cluster, dimension, tile), tile fastest, handed out through an atomic ticket so that an item only
// ever waits for items taken earlier (forward progress).  The running sums across the tiles of a segment come from a
// decoupled look-back: every tile publishes its aggregate, then walks back until it meets a published inclusive prefix.
// ---------------------------------------------------------------------------------------------------
struct __align__(16) AggSlot { Agg v; unsigned long long pad; };   // 32 bytes

// status words carry the epoch (level number + 1) of the search level that wrote them: words of earlier levels read as empty, so the look-back arrays are
// cleared once per search and not once per level (nothing in a level depends on a host-side memset of a size only the device knows)
__device__ __forceinline__ Agg ld_cg_agg(const AggSlot* p)
{
	const uint4* q = reinterpret_cast<const uint4*>(p);
	uint4 x = __ldcg(q), y = __ldcg(q + 1);
	Agg r; r.a = x.x; r.b = x.y; r.c = x.z; r.d = x.w; r.e = (unsigned long long)y.x | ((unsigned long long)y.y << 32);
	return r;
}
__device__ __forceinline__ void st_cg_agg(AggSlot* p, const Agg& v)
{
	uint4* q = reinterpret_cast<uint4*>(p);
	__stcg(q, make_uint4(v.a, v.b, v.c, v.d));
	__stcg(q + 1, make_uint4((uint32_t)v.e, (uint32_t)(v.e >> 32), 0u, 0u));
}

// Decoupled look-back of warp 0 over the earlier tiles of a segment (items w - tile .. w - 1), split layout: publishes this tile's aggregate, walks
// back to the nearest published inclusive prefix, publishes its own inclusive prefix and returns the exclusive one.
__device__ __forceinline__ Agg agg_lookback(uint64_t w, uint32_t tile, const Agg& total, uint32_t* __restrict__ status, AggSlot* __restrict__ aggs,
                                            AggSlot* __restrict__ prefixes, uint32_t epoch, uint32_t* __restrict__ error_flag)
{
	const int ln = threadIdx.x & 31;
	Agg carry = agg_zero();
	if(tile > 0) {
		if(ln == 0) {
			st_cg_agg(&aggs[w], total);
			lb_split_publish(&status[w], LB_AGG, epoch);
		}
		const bool ok = lb_walk(w, tile, [&](uint64_t i) { return ld_volatile_u32(&status[i]); }, [&](uint32_t raw) { return lb_split_state(raw, epoch); },
		                        [&](uint32_t, uint64_t i, bool take, uint32_t first_prefix) {
			Agg v = lb_split_value<Agg>(i, take, (uint32_t)ln == first_prefix, aggs, prefixes, ld_cg_agg);
#pragma unroll
			for(int o = 16; o > 0; o >>= 1) {
				Agg t2;
				t2.a = __shfl_xor_sync(0xffffffffu, v.a, o); t2.b = __shfl_xor_sync(0xffffffffu, v.b, o);
				t2.c = __shfl_xor_sync(0xffffffffu, v.c, o); t2.d = __shfl_xor_sync(0xffffffffu, v.d, o);
				t2.e = __shfl_xor_sync(0xffffffffu, v.e, o);
				v = agg_add(v, t2);
			}
			carry = agg_add(carry, v);
		});
		if(!ok && ln == 0)
			atomicExch(error_flag, 1u);
	}
	if(ln == 0) {
		st_cg_agg(&prefixes[w], agg_add(carry, total));
		lb_split_publish(&status[w], LB_PREFIX, epoch);
	}
	return carry;
}

// per-element contribution to the running sums of the split-scafs sweep (see the table in DESIGN.md section 3)
// a: ndps_in_scafs_that_belong of side 1, b: scafs_in of side 1, c: decrease of ndps_in_scafs_that_belong of side 2, d: decrease of scafs_in of side 2
__device__ __forceinline__ Agg contribution(uint32_t el, bool in_range, const ScafRow* __restrict__ rows, double fraction_in)
{
	const uint32_t cls = (el >> EL_CLASS_SHIFT) & 3u, aux = (el >> EL_AUX_SHIFT) & 3u;
	Agg x = agg_zero();
	if(cls == 2u)
		x.a = 1;
	if(aux == 0u && in_range)
		x.c = 1;
	if(cls == 1u || aux == 1u) {
		const uint4 r = __ldg(reinterpret_cast<const uint4*>(rows + (el & EL_SCAF_MASK)));
		const uint32_t r1 = (uint32_t)ceil(__dmul_rn(fraction_in, (double)r.x));
		if(cls == 1u) { x.a = r1; x.b = 1; }
		if(aux == 1u) { x.c = r1; x.d = 1; }
	}
	return x;
}

template <int STRATEGY>
__device__ __forceinline__ void block_best_out(CandRec best, uint32_t d, CandRec* sm_best, CandRec* __restrict__ out, uint64_t w)
{
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	if(__syncthreads_or(best.found)) {
#pragma unroll
		for(int o = 16; o > 0; o >>= 1) {
			CandRec other;
			other.k1 = __shfl_xor_sync(0xffffffffu, best.k1, o); other.k2 = __shfl_xor_sync(0xffffffffu, best.k2, o);
			other.p = __shfl_xor_sync(0xffffffffu, best.p, o); other.i0 = __shfl_xor_sync(0xffffffffu, best.i0, o);
			other.i1 = __shfl_xor_sync(0xffffffffu, best.i1, o); other.i2 = __shfl_xor_sync(0xffffffffu, best.i2, o);
			other.found = __shfl_xor_sync(0xffffffffu, best.found, o); other.dim0 = d;
			if(cand_better<STRATEGY>(other, best))
				best = other;
		}
		if(lane == 0)
			sm_best[warp] = best;
		__syncthreads();
		if(threadIdx.x == 0) {
			CandRec b = sm_best[0];
			for(int w2 = 1; w2 < SW_THREADS / 32; w2++)
				if(cand_better<STRATEGY>(sm_best[w2], b))
					b = sm_best[w2];
			out[w] = b;
		}
	}
	else if(threadIdx.x == 0)
		out[w] = best;
}

__global__ void __launch_bounds__(SW_THREADS, 3) k_sweep_split_scafs(const uint32_t* __restrict__ E, uint64_t N, const LevelCluster* __restrict__ clusters, uint32_t D,
                                                                    LevelCtl* __restrict__ ctl, const uint2* __restrict__ tile_tab, const ScafRow* __restrict__ rows,
                                                                    SweepParams prm, uint32_t epoch, uint32_t* __restrict__ status, AggSlot* __restrict__ aggs,
                                                                    AggSlot* __restrict__ prefixes, CandRec* __restrict__ out)
{
	__shared__ Agg sm_agg[SW_THREADS / 32 + 1];
	__shared__ CandRec sm_best[SW_THREADS / 32];
	__shared__ unsigned long long sm_w;
	__shared__ Agg sm_carry;
	const uint32_t TT = ctl->TT;
	const uint64_t items = (uint64_t)TT * D;
	// work items are (dimension, tile-table entry), entry fastest: the tiles of a (cluster, dimension) segment are consecutive items.  CTAs take items
	// through a ticket until none is left, so an item only ever waits for items taken earlier by CTAs that are running (forward progress).
	while(true) {
		if(threadIdx.x == 0)
			sm_w = atomicAdd(&ctl->tickets[1], 1ull);
		__syncthreads();
		const uint64_t w = sm_w;
		if(w >= items)
			break;
		const uint32_t d = (uint32_t)(w / TT);
		const uint2 te = __ldg(tile_tab + (uint32_t)(w - (uint64_t)d * TT));
		const uint32_t c = te.x, tile = te.y;
		const ClusterDesc cl = clusters[c].d;
		const uint32_t* __restrict__ seg = E + (uint64_t)d * N + cl.off;
		const uint32_t n = cl.n;
		CandRec best;
		best.found = 0; best.k1 = 0; best.k2 = 0; best.p = 0; best.i0 = best.i1 = best.i2 = 0; best.dim0 = d;
		if(!cl.ss_ok) {        // uniform over the tiles of the cluster: nobody waits for these items
			if(threadIdx.x == 0)
				out[w] = best;
			__syncthreads();
			continue;
		}
		const uint32_t t0 = tile * SW_TILE;
		const uint32_t i0 = t0 + threadIdx.x * SW_ITEMS;
		uint32_t el[SW_ITEMS];
		if(i0 + SW_ITEMS <= n && ((reinterpret_cast<uintptr_t>(seg + i0) & 15) == 0)) {
			const uint4* p4 = reinterpret_cast<const uint4*>(seg + i0);
#pragma unroll
			for(int q = 0; q < SW_ITEMS / 4; q++) {
				const uint4 x = __ldg(p4 + q);
				el[4 * q] = x.x; el[4 * q + 1] = x.y; el[4 * q + 2] = x.z; el[4 * q + 3] = x.w;
			}
		}
		else {
#pragma unroll
			for(int j = 0; j < SW_ITEMS; j++)
				el[j] = (i0 + j < n)? __ldg(seg + i0 + j) : 0u;   // class 0, no boundary: contributes nothing
		}
		// per-element contributions (recomputed in the candidate pass instead of being kept in registers)
		Agg tsum = agg_zero();
#pragma unroll
		for(int j = 0; j < SW_ITEMS; j++)
			tsum = agg_add(tsum, contribution(el[j], i0 + j < n, rows, prm.fraction_in));
		Agg total;
		Agg ex = block_excl_scan_agg(tsum, total, sm_agg);
		// decoupled look-back over the earlier tiles of this (cluster, dimension)
		if(threadIdx.x < 32) {
			const Agg carry = agg_lookback(w, tile, total, status, aggs, prefixes, epoch, &ctl->error);
			if(threadIdx.x == 0)
				sm_carry = carry;
		}
		__syncthreads();
		ex = agg_add(ex, sm_carry);
		// candidates: a boundary before element i means "all dps with value <= value[i-1]" is a threshold with p = i
#pragma unroll
		for(int j = 0; j < SW_ITEMS; j++) {
			const uint32_t p = i0 + j;
			if((el[j] & EL_BOUNDARY) && p < n && p >= prm.thr && n - p >= prm.thr) {
				// ...SplitScafs.cpp:131-154
				const uint32_t belong1 = ex.a, in1 = ex.b, belong2 = n - ex.c, in2 = cl.U - ex.d;
				if(belong1 >= prm.thr && belong2 >= prm.thr) {
					const uint32_t separated = cl.U - in1 - in2;
					const uint32_t in_small = (p < n - p)? in1 : in2, in_large = (p < n - p)? in2 : in1;
					const double ratio = __ddiv_rn((double)separated, (double)(int)in_small);
					double csr = __ddiv_rn((double)(int)in_small, (double)(int)in_large);
					if(csr < 1)
						csr = __ddiv_rn(1.0, csr);
					if(!best.found || ratio < best.k1 || (ratio == best.k1 && csr < best.k2)) {
						best.found = 1; best.k1 = ratio; best.k2 = csr; best.p = p; best.i0 = separated; best.i1 = in_small; best.i2 = in_large;
					}
				}
			}
			ex = agg_add(ex, contribution(el[j], i0 + j < n, rows, prm.fraction_in));
		}
		block_best_out<ABW_SPLIT_SCAFS>(best, d, sm_best, out, w);
		__syncthreads();
	}
}

// ---------------------------------------------------------------------------------------------------
// sens/spec sweep, second formulation.  Only the class-1 ("flip") elements carry per-scaffold quantities (T/2+1, T, n, SCG flag,
// length); everything a candidate needs is therefore a function of two COUNTS at its position -- class-2 elements before it and
// flip elements before it -- plus a table of prefix sums indexed by the flip count.  Those tables are built once per level
// from the per-dimension flip list (k_flip_prefix), where the per-scaffold gathers are a plain parallel stream; the sweep itself
// then never looks at a scaffold id: a warp reads 32 rows of 32 consecutive elements (coalesced 128-byte requests), turns the
// three flag bits of every row into ballot masks, and lane r keeps the masks of row r -- i.e. of 32 CONSECUTIVE elements.  Counts
// before any position are popcounts; the block scan and the look-back carry two small integers instead of five sums.
// ---------------------------------------------------------------------------------------------------
constexpr int SW_WARP_CHUNK = 32 * 32;            // elements per warp: 32 rows of 32

// payload of the sweep's packed look-back word (lb_pack): two counts below 2^28 (a problem holds fewer than 2^28 datapoints)
__device__ __forceinline__ unsigned long long cnt_payload(uint32_t nf, uint32_t nc) { return (unsigned long long)nf | ((unsigned long long)nc << 28); }

// Tables of a level, per (cluster, dimension), indexed by the number k of flip elements already passed:
//   F8[k-1]  = sums over the first k flips: x = T/2+1 (TP brought by the flips), y = T;  FC[k-1] = n (only kept when some scaffold has n < T)
//   scg_k[i] = k at which the i-th SCG-carrying scaffold flips (the SCG count of a candidate is a binary search in it)
//   klo, khi = the range of k for which both sides are >= scg_min_size bases long (ClusterQuality.cpp:118-120); lengths only matter through that test
// Tiles of FP_TILE list entries, items (dimension, tile-table entry) handed out by ticket, running sums across tiles by look-back.
constexpr int FP_ITEMS = 8;
constexpr int FP_TILE = SW_THREADS * FP_ITEMS;
// The per-scaffold records of a tile are staged in shared memory (coalesced list reads, the gathers of all eight entries of a thread in flight,
// 16-byte slots swizzled so that both the strided stores and the blocked loads are conflict free) instead of living in registers across the
// scan and the look-back: 40 registers instead of 128, six CTAs per SM instead of two.
// Resident CTAs per SM of the three look-back kernels of a sens/spec search level, measured on B200 (cfg2, 13 levels; registers are capped accordingly and a few values spill):
//   k_partition2 3 -> 4: 1625 -> 1500 us;  k_sweep_ss 4 -> 5 -> 6: 1222 -> 1159 -> 1135 us;  k_flip_prefix 4 -> 5 -> 6: 1150 -> 1088 -> 1217 us
constexpr int FLIP_CTAS = 5, SWEEP_CTAS = 6, PART_CTAS = 4;
__global__ void __launch_bounds__(SW_THREADS, FLIP_CTAS) k_flip_prefix(const uint32_t* __restrict__ flip_list, uint64_t Sf, const LevelCluster* __restrict__ clusters, uint32_t D,
                                                              LevelCtl* __restrict__ ctl, const uint2* __restrict__ ftile_tab, const uint4* __restrict__ frow,
                                                              uint32_t epoch, uint32_t* __restrict__ status, AggSlot* __restrict__ aggs,
                                                              AggSlot* __restrict__ prefixes, uint2* __restrict__ F8, uint32_t* __restrict__ FC, uint32_t* __restrict__ scg_k,
                                                              uint64_t Kstride, uint2* __restrict__ klohi, uint32_t Cstride, unsigned long long scg_min_size)
{
	__shared__ uint4 sm_r[FP_TILE];                        // {T (0: no entry), n | SCG flag << 31, length}
	__shared__ Agg sm_agg[SW_THREADS / 32];
	__shared__ unsigned long long sm_w;
	__shared__ Agg sm_carry;
	const uint32_t FTT = ctl->FPT;
	const uint64_t items = (uint64_t)FTT * D;
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	while(true) {
		if(threadIdx.x == 0)
			sm_w = atomicAdd(&ctl->tickets[0], 1ull);
		__syncthreads();
		const uint64_t w = sm_w;
		if(w >= items)
			break;
		const uint32_t d = (uint32_t)(w / FTT);
		const uint2 te = __ldg(ftile_tab + (uint32_t)(w - (uint64_t)d * FTT));
		const uint32_t tile = te.y;
		const uint32_t nf = clusters[te.x].d.nf, fOff = clusters[te.x].d.fOff;
		const uint64_t base = (uint64_t)d * Sf + fOff;
		const uint32_t* __restrict__ list = flip_list + base;
		{
			uint32_t sc[FP_ITEMS];
#pragma unroll
			for(int j = 0; j < FP_ITEMS; j++) {
				const uint32_t idx = tile * FP_TILE + j * SW_THREADS + threadIdx.x;
				sc[j] = (idx < nf)? (__ldg(list + idx) & EL_SCAF_MASK) : 0xFFFFFFFFu;      // a partition pass may have left a flag bit on the entry
			}
#pragma unroll
			for(int j = 0; j < FP_ITEMS; j++) {
				uint4 r = make_uint4(0, 0, 0, 0);
				if(sc[j] != 0xFFFFFFFFu)
					r = __ldg(frow + sc[j]);
				const uint32_t e = j * SW_THREADS + threadIdx.x;
				sm_r[e ^ ((e >> 3) & 7u)] = r;
			}
		}
		__syncthreads();
		const uint32_t e0 = threadIdx.x * FP_ITEMS, swz = threadIdx.x & 7u;     // this thread's eight consecutive entries
		Agg tsum = agg_zero();
#pragma unroll
		for(int j = 0; j < FP_ITEMS; j++) {
			const uint4 r = sm_r[e0 + ((uint32_t)j ^ swz)];
			if(r.x) {
				tsum.a += r.x / 2 + 1;         // the flip element brings itself and the floor(T/2) earlier dps of the scaffold (...Specificity.cpp:41-57)
				tsum.b += r.x;
				tsum.c += r.y & 0x7FFFFFFFu;
				tsum.d += r.y >> 31;
				tsum.e += (unsigned long long)r.z | ((unsigned long long)r.w << 32);
			}
		}
		Agg incl = tsum;
#pragma unroll
		for(int o = 1; o < 32; o <<= 1) {
			const Agg t = agg_shfl_up(incl, o);
			if(lane >= o)
				incl = agg_add(incl, t);
		}
		if(lane == 31)
			sm_agg[warp] = incl;
		__syncthreads();
		Agg wex = agg_zero(), total = agg_zero();
#pragma unroll
		for(int w2 = 0; w2 < SW_THREADS / 32; w2++) {
			const Agg t = sm_agg[w2];
			if(w2 < warp)
				wex = agg_add(wex, t);
			total = agg_add(total, t);
		}
		if(threadIdx.x < 32) {
			const Agg carry = agg_lookback(w, tile, total, status, aggs, prefixes, epoch, &ctl->error);
			if(threadIdx.x == 0)
				sm_carry = carry;
		}
		__syncthreads();
		Agg run = agg_add(agg_add(sm_carry, wex), incl);
		run.a -= tsum.a; run.b -= tsum.b; run.c -= tsum.c; run.d -= tsum.d; run.e -= tsum.e;
		const uint32_t kOff = clusters[te.x].d.kOff;
		const unsigned long long totLen = clusters[te.x].d.totLen;
		const uint32_t i0 = tile * FP_TILE + e0;
#pragma unroll
		for(int j = 0; j < FP_ITEMS; j++) {
			const uint4 r = sm_r[e0 + ((uint32_t)j ^ swz)];
			if(r.x) {
				const unsigned long long e_before = run.e;
				run.a += r.x / 2 + 1;
				run.b += r.x;
				run.c += r.y & 0x7FFFFFFFu;
				run.e += (unsigned long long)r.z | ((unsigned long long)r.w << 32);
				const uint32_t k = i0 + j + 1;                  // flips passed once this one is
				F8[base + i0 + j] = make_uint2(run.a, run.b);
				if(FC != nullptr)
					FC[base + i0 + j] = run.c;
				if(r.y >> 31) {
					run.d++;
					scg_k[(uint64_t)d * Kstride + kOff + run.d - 1] = k;
				}
				// lengths are non-decreasing in k: exactly one flip crosses each limit
				if(e_before < scg_min_size && run.e >= scg_min_size)
					klohi[(uint64_t)d * Cstride + te.x].x = k;
				if(totLen >= scg_min_size && e_before <= totLen - scg_min_size && run.e > totLen - scg_min_size)
					klohi[(uint64_t)d * Cstride + te.x].y = k - 1;
			}
		}
		__syncthreads();
	}
}

__global__ void __launch_bounds__(SW_THREADS, SWEEP_CTAS) k_sweep_ss(const uint32_t* __restrict__ E, uint64_t N, const LevelCluster* __restrict__ clusters, uint32_t D,
                                                           LevelCtl* __restrict__ ctl, const uint2* __restrict__ tile_tab, const uint2* __restrict__ F8,
                                                           const uint32_t* __restrict__ FC, const uint32_t* __restrict__ scg_k, uint64_t Kstride,
                                                           const uint2* __restrict__ klohi, uint32_t Cstride, uint64_t Sf, const uint8_t* __restrict__ pass_tab,
                                                           SweepParams prm, uint32_t epoch, unsigned long long* __restrict__ lookback, CandRec* __restrict__ out)
{
	__shared__ uint32_t sm_warp[SW_THREADS / 32];
	__shared__ CandRec sm_best[SW_THREADS / 32];
	__shared__ unsigned long long sm_w;
	__shared__ uint32_t sm_carry[2];
	const uint32_t TT = ctl->TT;
	const uint64_t items = (uint64_t)TT * D, tab_stride = ctl->tab_total;
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	while(true) {
		if(threadIdx.x == 0)
			sm_w = atomicAdd(&ctl->tickets[1], 1ull);
		__syncthreads();
		const uint64_t w = sm_w;
		if(w >= items)
			break;
		const uint32_t d = (uint32_t)(w / TT);
		const uint2 te = __ldg(tile_tab + (uint32_t)(w - (uint64_t)d * TT));
		const uint32_t tile = te.y;
		const ClusterDesc cl = clusters[te.x].d;
		const uint32_t* __restrict__ seg = E + (uint64_t)d * N + cl.off;
		const uint32_t n = cl.n;
		const uint32_t wbase = tile * SW_TILE + warp * SW_WARP_CHUNK;
		// 32 coalesced rows; lane r ends up with the flag masks of row r = elements [wbase + 32 r, wbase + 32 r + 32)
		uint32_t mF = 0, mC = 0, mB = 0;
		if(wbase < n) {
			uint32_t el[32];
			if(wbase + SW_WARP_CHUNK <= n) {                    // warp uniform: the whole chunk exists
#pragma unroll
				for(int r = 0; r < 32; r++)
					el[r] = __ldg(seg + wbase + r * 32 + lane);
			}
			else {
#pragma unroll
				for(int r = 0; r < 32; r++) {
					const uint32_t idx = wbase + r * 32 + lane;
					el[r] = (idx < n)? __ldg(seg + idx) : 0u;      // class 0, no boundary: contributes nothing
				}
			}
#pragma unroll
			for(int r = 0; r < 32; r++) {
				const uint32_t f = __ballot_sync(0xffffffffu, el[r] & EL_FLIP_BIT);
				const uint32_t c2 = __ballot_sync(0xffffffffu, el[r] & EL_CLS2_BIT);
				const uint32_t b = __ballot_sync(0xffffffffu, el[r] & EL_BOUNDARY);
				if(lane == r) { mF = f; mC = c2; mB = b; }
			}
		}
		const uint32_t i0 = wbase + lane * 32;                  // first element of this thread's row
		// exclusive block scan of (flip count, class-2 count), 16 bits each: a tile holds 8192 elements
		const uint32_t mine = __popc(mF) | (__popc(mC) << 16);
		uint32_t incl = mine;
#pragma unroll
		for(int o = 1; o < 32; o <<= 1) {
			const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
			if(lane >= o)
				incl += t;
		}
		if(lane == 31)
			sm_warp[warp] = incl;
		__syncthreads();
		uint32_t wex = 0, btot = 0;
#pragma unroll
		for(int w2 = 0; w2 < SW_THREADS / 32; w2++) {
			const uint32_t t = sm_warp[w2];
			if(w2 < warp)
				wex += t;
			btot += t;
		}
		const uint32_t ex = wex + incl - mine;
		// decoupled look-back over the earlier tiles of this (cluster, dimension)
		if(threadIdx.x < 32) {
			const uint32_t totF = btot & 0xFFFFu, totC = btot >> 16;
			uint32_t cF = 0, cC = 0;
			if(tile > 0) {
				if(lane == 0)
					st_volatile_u64(&lookback[w], lb_pack(cnt_payload(totF, totC), LB_AGG, epoch));
				const bool ok = lb_walk(w, tile, [&](uint64_t i) { return ld_volatile_u64(&lookback[i]); },
				                        [&](unsigned long long v) { return lb_packed_state(v, epoch); },
				                        [&](unsigned long long v, uint64_t, bool take, uint32_t) {
					cF += __reduce_add_sync(0xffffffffu, take? (uint32_t)(v & 0xFFFFFFFull) : 0u);
					cC += __reduce_add_sync(0xffffffffu, take? (uint32_t)((v >> 28) & 0xFFFFFFFull) : 0u);
				});
				if(!ok && lane == 0)
					atomicExch(&ctl->error, 1u);
			}
			if(lane == 0) {
				st_volatile_u64(&lookback[w], lb_pack(cnt_payload(cF + totF, cC + totC), LB_PREFIX, epoch));
				sm_carry[0] = cF;
				sm_carry[1] = cC;
			}
		}
		__syncthreads();
		const uint32_t nF0 = sm_carry[0] + (ex & 0xFFFFu), nC0 = sm_carry[1] + (ex >> 16);
		// candidates: a boundary before element i means "all dps with value <= value[i-1]" is a threshold with p = i
		CandRec best;
		best.found = 0; best.k1 = 0; best.k2 = 0; best.p = 0; best.i0 = best.i1 = best.i2 = 0; best.dim0 = d;
		const uint8_t* __restrict__ tab = pass_tab + (uint64_t)d * tab_stride + cl.tabOff;
		const uint64_t fbase = (uint64_t)d * Sf + cl.fOff;
		const uint32_t* __restrict__ sk = scg_k + (uint64_t)d * Kstride + cl.kOff;
		uint32_t bm = mB, lastk = 0;
		uint2 f = make_uint2(0, 0);
		uint32_t fc = 0;
		while(bm) {
			const int j = __ffs(bm) - 1;
			bm &= bm - 1;
			const uint32_t p = i0 + j;                          // p < n: elements past the end have no boundary bit
			if(p < prm.thr || n - p < prm.thr)
				continue;
			const uint32_t lt = (1u << j) - 1u;
			const uint32_t k = nF0 + __popc(mF & lt);
			if(k != lastk) {
				f = __ldg(F8 + fbase + k - 1);                  // k == 0 only before the first reload: f is zero then
				fc = (FC != nullptr)? __ldg(FC + fbase + k - 1) : f.y;     // n == T for every scaffold unless the caller passed partial scaffolds
				lastk = k;
			}
			const uint32_t a = nC0 + __popc(mC & lt) + f.x;     // TP1
			// ...Specificity.cpp:146-161 with TP1/FP1/TP2/FP2 written as prefix sums
			uint32_t TP, tot, u;
			if(p < n - p) { TP = a; tot = f.y; u = p; }
			else { TP = (n - p) - (fc - a); tot = cl.totT - f.y; u = n - p; }
			if(tot == 0)
				continue;
			const float fTP = (float)TP;
			if(!(fTP >= prm.prune * (float)tot && fTP >= prm.prune * (float)u))
				continue;
			const double sens = __ddiv_rn((double)(int)TP, (double)(int)tot), spec = __ddiv_rn((double)(int)TP, (double)(int)u);
			const double score = __dmul_rn(sens, spec);
			if(score >= prm.min_score && (!best.found || score > best.k1)) {
				// SCG-carrying scaffolds among the first k flips: the entries of scg_k (increasing) that are <= k
				uint32_t lo = 0, hi = cl.K;
				while(lo < hi) {
					const uint32_t mid = (lo + hi) >> 1;
					if(__ldg(sk + mid) <= k) lo = mid + 1; else hi = mid;
				}
				const uint8_t pt = tab[lo];
				bool ok = (pt == 1);
				if(pt == 2) {
					const uint2 kk = __ldg(klohi + (uint64_t)d * Cstride + te.x);
					ok = k >= kk.x && k <= kk.y;                // both sides at least scg_min_size bases long
				}
				if(ok) {
					best.found = 1; best.k1 = score; best.p = p; best.i0 = TP; best.i1 = tot; best.i2 = u;
				}
			}
		}
		block_best_out<ABW_SENS_SPEC>(best, d, sm_best, out, w);
		__syncthreads();
	}
}

// best candidate of every cluster over its (dimension, tile) items: the reference's total order
// (score, then lowest dimension, then lowest value; ...Specificity.cpp:137-140 under the mutex, ClusterSeparator.cpp:11-16)
constexpr int RB_THREADS = 1024;       // one CTA per cluster: the first levels have few clusters with thousands of candidates each (level 0 of cfg2: 5292), so the
                                       // time of this kernel is the number of dependent load rounds per thread (256 threads: 22 us at level 0)
template <int STRATEGY>
__global__ void __launch_bounds__(RB_THREADS) k_reduce_best(const CandRec* __restrict__ per_item, uint32_t D, const LevelCtl* __restrict__ ctl,
                                                    const LevelCluster* __restrict__ clusters, uint32_t dim_offset, uint32_t dim_stride, CandRec* __restrict__ out)
{
	__shared__ CandRec sm[RB_THREADS];
	const uint32_t C = ctl->C, TT = ctl->TT;
	for(uint32_t c = blockIdx.x; c < C; c += gridDim.x) {
		const uint32_t tiles = (clusters[c].d.n + SW_TILE - 1) / SW_TILE, tile0 = clusters[c].d.tile0;
		CandRec best;
		best.found = 0; best.k1 = best.k2 = 0; best.p = 0; best.i0 = best.i1 = best.i2 = 0; best.dim0 = 0;
		const uint32_t total = D * tiles;                     // below 2^31: abw_search_run checks the number of (dimension, tile) items of a level
		for(uint32_t i = threadIdx.x; i < total; i += blockDim.x) {
			const uint32_t d = i / tiles, t = i - d * tiles;
			CandRec x = per_item[(uint64_t)d * TT + tile0 + t];
			x.dim0 = d;
			if(cand_better<STRATEGY>(x, best))
				best = x;
		}
		sm[threadIdx.x] = best;
		__syncthreads();
		for(uint32_t s2 = blockDim.x / 2; s2 > 0; s2 >>= 1) {
			if(threadIdx.x < s2 && cand_better<STRATEGY>(sm[threadIdx.x + s2], sm[threadIdx.x]))
				sm[threadIdx.x] = sm[threadIdx.x + s2];
			__syncthreads();
		}
		if(threadIdx.x == 0) {
			CandRec b = sm[0];
			b.dim0 = b.dim0 * dim_stride + dim_offset;          // global dimension index from here on (a sharded search holds every dim_stride-th dimension)
			out[c] = b;
		}
		__syncthreads();
	}
}

// ---------------------------------------------------------------------------------------------------
// SCG acceptance table, ClusterQuality.cpp:96-136 + SCGdb.cpp:21-38.  One CTA per (cluster, dimension).
// entry k (k SCG-carrying scaffolds already assigned to side 1): 0 reject, 1 accept, 2 decide on the sizes.
// ---------------------------------------------------------------------------------------------------
constexpr int PT_WARPS = 8;
// the K events are cut into PT_WARPS chunks; a first pass ORs the masks of every chunk, then every warp
// runs the suffix and prefix passes over its own chunk, seeded with the ORs of the chunks after / before it
__global__ void __launch_bounds__(PT_WARPS * 32) k_pass_table(const uint32_t* __restrict__ scg_list, uint64_t list_stride, const LevelCluster* __restrict__ clusters,
                             const LevelCtl* __restrict__ ctl, const uint64_t* __restrict__ scgmask, uint32_t W, double overlap_thr, uint64_t* __restrict__ suffix_tmp,
                             uint8_t* __restrict__ tab, uint32_t D, uint2* __restrict__ klohi, uint32_t Cstride, unsigned long long scg_min_size)
{
	__shared__ unsigned long long chunk_or[PT_WARPS][SCG_WMAX];
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	const uint32_t C = ctl->C;
	const uint64_t tab_stride = ctl->tab_total, items = (uint64_t)C * D;
	for(uint64_t item = blockIdx.x; item < items; item += gridDim.x) {
		const uint32_t c = (uint32_t)(item % C), d = (uint32_t)(item / C);
		const ClusterDesc cl = clusters[c].d;
		const unsigned long long* __restrict__ never_mask = clusters[c].never;
		if(threadIdx.x == 0)                               // size test of the level (k_flip_prefix narrows it): with no flip at all side 1 is empty
			klohi[(uint64_t)d * Cstride + c] = (cl.totLen >= scg_min_size)? make_uint2(scg_min_size == 0? 0u : 0xFFFFFFFFu, 0xFFFFFFFFu) : make_uint2(0xFFFFFFFFu, 0u);
		const uint32_t* __restrict__ list = scg_list + (uint64_t)d * list_stride + cl.kOff;
		uint64_t* __restrict__ suf = suffix_tmp + ((uint64_t)d * list_stride + cl.kOff) * W;     // suf[k] = OR of masks k..K-1
		uint8_t* __restrict__ t = tab + (uint64_t)d * tab_stride + cl.tabOff;
		const uint32_t K = cl.K;
		// entries 0..K (K+1 of them) and masks 0..K-1 share the chunk boundaries
		const uint32_t ech = ((K + 1 + PT_WARPS - 1) / PT_WARPS + 31u) & ~31u;
		const uint32_t e0 = min(K + 1, warp * ech), e1 = min(K + 1, e0 + ech);      // entries of this warp
		const uint32_t m1 = min(K, e1);                                            // its masks: [e0, m1)
		for(uint32_t w = 0; w < W; w++) {
			unsigned long long o = 0;
			for(uint32_t k = e0 + lane; k < m1; k += 32)
				o |= scgmask[(uint64_t)(list[k] & EL_SCAF_MASK) * W + w];
			o = (unsigned long long)__reduce_or_sync(0xffffffffu, (uint32_t)o) | ((unsigned long long)__reduce_or_sync(0xffffffffu, (uint32_t)(o >> 32)) << 32);
			if(lane == 0)
				chunk_or[warp][w] = o;
		}
		__syncthreads();
		if(e0 < e1) {
			// pass 1 (backwards): suffix ORs, one mask word at a time
			for(uint32_t w = 0; w < W; w++) {
				uint64_t carry = 0;
				for(int w2 = warp + 1; w2 < PT_WARPS; w2++)
					carry |= chunk_or[w2][w];
				for(int64_t base = (int64_t)e0 + (int64_t)((m1 > e0? m1 - e0 + 31 : 0) / 32) * 32 - 32; base >= (int64_t)e0; base -= 32) {
					const uint32_t k = (uint32_t)base + lane;
					uint64_t m = (k < m1)? scgmask[(uint64_t)(list[k] & EL_SCAF_MASK) * W + w] : 0ull;
#pragma unroll
					for(int o = 1; o < 32; o <<= 1) {
						uint64_t x = __shfl_down_sync(0xffffffffu, m, o);
						if(lane + o < 32)
							m |= x;
					}
					m |= carry;
					if(k < m1)
						suf[(uint64_t)k * W + w] = m;
					carry = __shfl_sync(0xffffffffu, m, 0);
				}
			}
			__syncwarp();
			// pass 2 (forwards): entry k sees side 1 = events [0, k), side 2 = events [k, K) plus the scaffolds that can never flip
			uint64_t carry[SCG_WMAX], after[SCG_WMAX];
#pragma unroll
			for(uint32_t w = 0; w < SCG_WMAX; w++) {
				carry[w] = 0;
				after[w] = 0;
				if(w < W) {
					for(int w2 = 0; w2 < warp; w2++)
						carry[w] |= chunk_or[w2][w];
					for(int w2 = warp + 1; w2 < PT_WARPS; w2++)
						after[w] |= chunk_or[w2][w];                    // suffix of an entry that lies past the masks of this chunk (k == m1)
				}
			}
			for(uint32_t base = e0; base < e1; base += 32) {
				const uint32_t k = base + lane;
				uint32_t g1 = 0, g2 = 0, g12 = 0;
#pragma unroll
				for(uint32_t w = 0; w < SCG_WMAX; w++) {
					if(w < W) {
						// mask of event k-1, unless it belongs to an earlier chunk (then it is already in the carry)
						uint64_t pre = (k >= 1 && k - 1 >= e0 && k - 1 < K)? scgmask[(uint64_t)(list[k - 1] & EL_SCAF_MASK) * W + w] : 0ull;
#pragma unroll
						for(int o = 1; o < 32; o <<= 1) {
							uint64_t x = __shfl_up_sync(0xffffffffu, pre, o);
							if(lane >= o)
								pre |= x;
						}
						pre |= carry[w];
						carry[w] = __shfl_sync(0xffffffffu, pre, 31);
						const uint64_t s2 = ((k < m1)? suf[(uint64_t)k * W + w] : after[w]) | never_mask[w];
						g1 += __popcll(pre);
						g2 += __popcll(s2);
						g12 += __popcll(pre & s2);
					}
				}
				if(k < e1) {
					uint8_t r;
					if(g1 == 0 || g2 == 0)
						r = 2;                                                  // ClusterQuality.cpp:118-120: decided on the two total sizes
					else
						r = (__ddiv_rn((double)g12, (double)min(g1, g2)) < overlap_thr)? 0 : 1;   // :130
					t[k] = r;
				}
			}
		}
		__syncthreads();
	}
}

// ---------------------------------------------------------------------------------------------------
// The work list on the device (abawaca.cpp:98-197, ClusterSeparator.cpp:25-54, 82-134).  Per level:
//   k_level_jobs    (one CTA)  merges the per-rank bests, applies is_legal, lists the clusters with a best separation ("jobs") and the work items of the next two kernels
//   k_count_low                datapoints of every scaffold on the low side of the separating value
//   k_scaf_sides               scaffold vote, re-homing, child statistics, separating value
//   k_level_decide  (one CTA)  >= 100 check, ids, records, the clusters of the next level with their tile tables, the partition plans, the terminal clusters
//   k_finalize_terminal        bins, total size and SCG tallies of the terminal clusters (its last CTA fills their records)
//   k_partition2               stable partition of scaffold list, elements, flip lists and SCG lists of the split clusters
// ---------------------------------------------------------------------------------------------------
struct SplitJob {
	uint32_t cluster;    // index into the level's cluster array
	uint32_t dim0;       // winning dimension (global index)
	uint32_t p;          // datapoints with value <= separating value
	uint32_t swapped;    // cluster1 is the high side (ClusterSeparator.cpp:49-53)
	uint32_t slot;       // index of the job in the level-wide (all ranks) job list: where its statistics go
	uint32_t sstar;      // scaffold of the last datapoint on the low side (set on the rank that holds the dimension): it carries the separating value
};

struct ChildStats {      // [job][2]; summed across ranks as 64-bit words in a sharded search (no 32-bit half can overflow)
	unsigned long long ndps, totLen;
	uint32_t ns, nassigned, totT, K, viol, nflip;
};

struct PartJob {
	uint64_t off;        // parent segment (child 1 is written at off, child 2 at off + n1)
	uint32_t n, n1;
};

struct TermJob { uint32_t sOff, ns, id, rec; };          // rec: index of the cluster's record (0xFFFFFFFF: none)
struct TermStats { unsigned long long total_size, scg_copies; };

constexpr int LV_THREADS = 1024;                            // the single-CTA kernels
constexpr uint32_t CL_CHUNK = 4096;                         // elements per work item of k_count_low
constexpr uint32_t SS_CHUNK = 128;                          // scaffolds per work item of k_scaf_sides
constexpr uint32_t TM_CHUNK = 512;                          // scaffolds per work item of k_finalize_terminal

// buffers of a search run that the level kernels share (device pointers; passed by value)
struct LevelBufs {
	LevelCtl* ctl;
	LevelProgress* prog;                                    // mapped pinned host memory
	LevelCluster* cl[2];
	CandRec *best, *best_all;                               // [Cmax] of this rank; [world][Cstride] gathered
	SplitJob* jobs;
	uint32_t *jobs_mine, *job_of;
	abw_best* bestrec;
	uint2 *cl_tab, *ss_tab, *tile_tab, *fp_tab, *part_tab, *tm_tab;
	PartJob* part_jobs;                                     // [4][Pmax]
	TermJob* tjobs;
	TermStats* tstats;
	uint64_t* tunion;
	abw_cluster_rec* recs;
	uint32_t rec_cap, Cmax, Pmax, pad;
	uint32_t* low;
};

// exclusive scan of one value per thread over a CTA of LV_THREADS threads; total = sum.  sm: uint32_t[33]
__device__ __forceinline__ uint32_t cta_excl_scan(uint32_t v, uint32_t& total, uint32_t* sm)
{
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	uint32_t incl = v;
#pragma unroll
	for(int o = 1; o < 32; o <<= 1) {
		const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
		if(lane >= o)
			incl += t;
	}
	if(lane == 31)
		sm[warp] = incl;
	__syncthreads();
	if(warp == 0) {
		const uint32_t w = sm[lane];
		uint32_t wi = w;
#pragma unroll
		for(int o = 1; o < 32; o <<= 1) {
			const uint32_t t = __shfl_up_sync(0xffffffffu, wi, o);
			if(lane >= o)
				wi += t;
		}
		sm[lane] = wi - w;
		if(lane == 31)
			sm[32] = wi;
	}
	__syncthreads();
	const uint32_t r = sm[warp] + incl - v;
	total = sm[32];
	__syncthreads();
	return r;
}

// entry i of n owns cnt(i) consecutive slots of a table: first(i, slot) is told where they start and, if tab is not null, tab[slot + t] = (i, t).
// Returns the number of slots.  Called by all LV_THREADS threads of the CTA.
template <class CountF, class FirstF>
__device__ __forceinline__ uint32_t cta_expand(uint32_t n, uint2* __restrict__ tab, CountF cnt, FirstF first, uint32_t* sm)
{
	uint32_t run = 0;
	for(uint32_t b = 0; b < n; b += LV_THREADS) {
		const uint32_t i = b + threadIdx.x;
		const uint32_t c = (i < n)? cnt(i) : 0u;
		uint32_t total;
		const uint32_t ex = cta_excl_scan(c, total, sm);
		if(i < n) {
			first(i, run + ex);
			if(tab != nullptr)
				for(uint32_t t = 0; t < c; t++)
					tab[run + ex + t] = make_uint2(i, t);
		}
		run += total;
	}
	return run;
}

__device__ __forceinline__ void best_reset(abw_best& b, int strategy)
{
	b.found = 0; b.dim = 0; b.value = -1; b.a = 0; b.b = 0; b.legal = 0;
	if(strategy == ABW_SPLIT_SCAFS) { b.a = 1000000; b.b = 1000000; }       // ClusteringResult::reset of the split-scafs strategy
}

__global__ void __launch_bounds__(LV_THREADS) k_level_jobs(const LevelBufs B, int cur, uint32_t world, uint32_t Cstride, int strategy, const abw_params prm,
                                                         uint32_t dim_offset, uint32_t dim_stride, uint32_t Dlocal, const uint32_t* __restrict__ E, uint64_t N,
                                                         ChildStats* __restrict__ stats, unsigned long long* __restrict__ value_key, uint64_t* __restrict__ child_never, uint32_t W)
{
	__shared__ uint32_t sm[33];
	__shared__ unsigned long long sm_el;
	LevelCtl* const ctl = B.ctl;
	const LevelCluster* __restrict__ cls = B.cl[cur];
	const uint32_t C = ctl->C;
	if(threadIdx.x == 0)
		sm_el = 0;
	__syncthreads();
	uint32_t J = 0;
	unsigned long long el = 0;
	for(uint32_t b0 = 0; b0 < C; b0 += LV_THREADS) {
		const uint32_t c = b0 + threadIdx.x;
		CandRec best;
		best.found = 0;
		if(c < C) {
			best = B.best[c];
			if(world > 1) {
				// the per-rank bests of the cluster, gathered: the same total order on every rank (ClusterSeparator.cpp:11-16)
				best = B.best_all[c];
				for(uint32_t r = 1; r < world; r++) {
					const CandRec x = B.best_all[(size_t)r * Cstride + c];
					if((strategy == ABW_SENS_SPEC)? cand_better<ABW_SENS_SPEC>(x, best) : cand_better<ABW_SPLIT_SCAFS>(x, best))
						best = x;
				}
			}
		}
		const bool found = c < C && best.found;
		uint32_t total;
		const uint32_t ex = cta_excl_scan(found? 1u : 0u, total, sm);
		if(c < C) {
			const uint32_t n = cls[c].d.n;
			el += (unsigned long long)n * Dlocal;
			abw_best hb;
			best_reset(hb, strategy);
			if(found) {
				hb.found = 1;
				hb.dim = best.dim0 + 1;
				if(strategy == ABW_SENS_SPEC) {
					// same IEEE operations as ClusterStats::get_sensitivity / get_specificity (...Specificity.h:74-75) and is_legal (:31-35)
					hb.a = __ddiv_rn((double)(int)best.i0, (double)(int)best.i1);
					hb.b = __ddiv_rn((double)(int)best.i0, (double)(int)best.i2);
					hb.legal = (hb.a >= prm.sensitivity_threshold) && (hb.b >= prm.specificity_threshold) && (__dadd_rn(hb.a, hb.b) >= prm.sum_threshold) &&
					           (__dmul_rn(hb.a, hb.b) >= prm.product_threshold);
				}
				else {
					hb.a = best.k1;
					hb.b = best.k2;
					hb.legal = hb.a <= prm.split_scaf_ratio_threshold;     // ...SplitScafs.h:38
				}
				SplitJob jb;
				jb.cluster = c; jb.dim0 = best.dim0; jb.p = best.p;
				jb.swapped = (n - best.p) < best.p;             // ClusterSeparator.cpp:49
				jb.slot = J + ex;
				jb.sstar = 0xFFFFFFFFu;
				B.jobs[J + ex] = jb;
				B.job_of[c] = J + ex;
			}
			else
				B.job_of[c] = 0xFFFFFFFFu;
			B.bestrec[c] = hb;
		}
		J += total;
	}
	__syncthreads();
	// jobs whose winning dimension lives on this rank (all of them when the search is not sharded)
	uint32_t JM = 0;
	for(uint32_t b0 = 0; b0 < J; b0 += LV_THREADS) {
		const uint32_t j = b0 + threadIdx.x;
		bool mine = false;
		if(j < J) {
			const uint32_t d = B.jobs[j].dim0;
			mine = d >= dim_offset && (d - dim_offset) % dim_stride == 0 && (d - dim_offset) / dim_stride < Dlocal;
		}
		uint32_t total;
		const uint32_t ex = cta_excl_scan(mine? 1u : 0u, total, sm);
		if(mine) {
			B.jobs_mine[JM + ex] = j;
			const SplitJob jb = B.jobs[j];
			B.jobs[j].sstar = E[(uint64_t)((jb.dim0 - dim_offset) / dim_stride) * N + cls[jb.cluster].d.off + jb.p - 1] & EL_SCAF_MASK;   // p >= 1: a candidate has datapoints on both sides
		}
		JM += total;
	}
	__syncthreads();
	const uint32_t cl_items = cta_expand(JM, B.cl_tab, [&](uint32_t k) { return (B.jobs[B.jobs_mine[k]].p + CL_CHUNK - 1) / CL_CHUNK; }, [](uint32_t, uint32_t) {}, sm);
	const uint32_t ss_items = cta_expand(JM, B.ss_tab, [&](uint32_t k) { return (cls[B.jobs[B.jobs_mine[k]].cluster].d.ns + SS_CHUNK - 1) / SS_CHUNK; },
	                                     [](uint32_t, uint32_t) {}, sm);
	for(uint32_t i = threadIdx.x; i < 2 * J; i += LV_THREADS) {
		ChildStats z;
		z.ndps = 0; z.totLen = 0; z.ns = z.nassigned = z.totT = z.K = z.viol = z.nflip = 0;
		stats[i] = z;
	}
	for(uint32_t i = threadIdx.x; i < J; i += LV_THREADS)
		value_key[i] = 0;
	for(uint32_t i = threadIdx.x; i < 2 * J * W; i += LV_THREADS)
		child_never[i] = 0;
	atomicAdd(&sm_el, el);
	__syncthreads();
	if(threadIdx.x == 0) {
		ctl->J = J; ctl->JM = JM; ctl->CL_items = cl_items; ctl->SS_items = ss_items;
		ctl->sweep_elements += sm_el;
		if(C > 0)
			ctl->sweep_launches++;
	}
}

__global__ void __launch_bounds__(256) k_count_low(const uint32_t* __restrict__ E, uint64_t N, const LevelBufs B, int cur, uint32_t dim_offset, uint32_t dim_stride,
                                                  uint32_t* __restrict__ low)
{
	const LevelCluster* __restrict__ cls = B.cl[cur];
	const uint32_t items = B.ctl->CL_items;
	for(uint32_t it = blockIdx.x; it < items; it += gridDim.x) {
		const uint2 te = B.cl_tab[it];
		const SplitJob jb = B.jobs[B.jobs_mine[te.x]];
		const uint32_t* __restrict__ seg = E + (uint64_t)((jb.dim0 - dim_offset) / dim_stride) * N + cls[jb.cluster].d.off;
		const uint32_t i0 = te.y * CL_CHUNK, i1 = min(jb.p, i0 + CL_CHUNK);
		for(uint32_t i = i0 + threadIdx.x; i < i1; i += blockDim.x)
			atomicAdd(&low[seg[i] & EL_SCAF_MASK], 1u);
	}
}

// Where the value of (datapoint, dimension) lives: the caller's matrix, in the caller's layout, read in place (no column-major copy is made).
struct ValSrc {
	const double*   p;
	uint64_t        ld;
	int             layout;
	const uint64_t* rowidx;        // matrix row of every datapoint (device), or null: datapoint i is row i
};
__device__ __forceinline__ double val_at(const ValSrc& v, uint64_t dp, uint32_t d)
{
	const uint64_t r = v.rowidx? v.rowidx[dp] : dp;
	if(v.layout == ABW_LAYOUT_ROWMAJOR_MILLI32)            // integer thousandths: the value is the double abawaca-build printed, int(1000 x) / 1000.0
		return __ddiv_rn((double)reinterpret_cast<const uint32_t*>(v.p)[r * v.ld + d], 1000.0);
	return (v.layout == ABW_LAYOUT_ROWMAJOR)? v.p[r * v.ld + d] : v.p[(uint64_t)d * v.ld + r];
}

__device__ __forceinline__ unsigned long long orderable(double v)
{
	v = v + 0.0;                                    // -0.0 and +0.0 compare equal in comp_by_value (ClusterSeparator.cpp:8)
	unsigned long long b = (unsigned long long)__double_as_longlong(v);
	return (b >> 63)? ~b : (b | 0x8000000000000000ull);
}
// one thread per scaffold of every cluster with a best separation: vote (ClusterSeparator.cpp:94-101), child statistics; the first warp of a job's first item
// recovers the separating value.  The statistics of a warp are combined before they reach the two counters of the job (one atomic per warp and field).
// low[] is cleared on the way (the entry of the scaffold that carries the separating value by k_level_decide).
__global__ void __launch_bounds__(SS_CHUNK) k_scaf_sides(const uint32_t* __restrict__ scaf_list, const LevelBufs B, int cur, uint32_t dim_offset, uint32_t dim_stride,
                             const ScafRow* __restrict__ rows, uint32_t* __restrict__ low, const uint64_t* __restrict__ dp_first, const ValSrc vsrc,
                             const uint64_t* __restrict__ scgmask, uint32_t W, int strategy, double fraction_in, uint8_t* __restrict__ side, uint8_t* __restrict__ new_assigned,
                             ChildStats* __restrict__ stats, uint64_t* __restrict__ child_never, unsigned long long* __restrict__ value_key)
{
	const LevelCluster* __restrict__ cls = B.cl[cur];
	const uint32_t items = B.ctl->SS_items;
	const int lane = threadIdx.x & 31;
	for(uint32_t it = blockIdx.x; it < items; it += gridDim.x) {
		const uint2 te = B.ss_tab[it];
		const SplitJob jb = B.jobs[B.jobs_mine[te.x]];
		const ClusterDesc cl = cls[jb.cluster].d;
		if(te.y == 0 && threadIdx.x < 32) {
			// separating value = largest value on the low side = value of the datapoint at position p - 1 of the winning dimension; that datapoint belongs to
			// scaffold sstar and is its lo-th smallest (the sort is stable and the datapoints of a scaffold are consecutive: ties go by datapoint index)
			const uint32_t s = jb.sstar;
			const ScafRow r = rows[s];
			const uint32_t lo = low[s];
			const uint64_t f = dp_first[s];
			const uint32_t dl = (jb.dim0 - dim_offset) / dim_stride;
			unsigned long long kth = 0;
			for(uint32_t a = lane; a < r.n; a += 32) {
				const unsigned long long ka = orderable(val_at(vsrc, f + a, dl));
				uint32_t rank = 0;
				for(uint32_t b = 0; b < r.n; b++) {
					const unsigned long long kb = orderable(val_at(vsrc, f + b, dl));
					rank += (kb < ka) || (kb == ka && b < a);
				}
				if(rank + 1 == lo)
					kth = ka;
			}
#pragma unroll
			for(int o = 16; o > 0; o >>= 1)
				kth = max(kth, __shfl_xor_sync(0xffffffffu, kth, o));
			if(lane == 0)
				value_key[jb.slot] = kth;
		}
		const uint32_t i = te.y * SS_CHUNK + threadIdx.x;
		const bool active = i < cl.ns;
		uint32_t sd = 0, rn = 0, rT = 0;
		unsigned long long rlen = 0;
		bool assigned_any = false, flippable = false, has_scg = false, viol = false;
		if(active) {
			const uint32_t s = scaf_list[cl.sOff + i] & EL_SCAF_MASK;      // the partition kernel leaves its flag bit on list entries
			const ScafRow r = rows[s];
			const uint32_t lo = low[s];
			if(s != jb.sstar)
				low[s] = 0;
			const uint32_t c1 = jb.swapped? r.n - lo : lo, c2 = r.n - c1;
			const bool A1 = c1 > 0 && 2ull * c1 >= r.T;          // :95-97
			const bool A2 = c2 > 0 && 2ull * c2 > r.T;           // :98-101
			// dps not in a scaffold assigned to cluster2 end up in cluster1 (:104-122)
			sd = A2? 2u : 1u;
			side[s] = (uint8_t)sd;
			new_assigned[s] = A1? 1 : (A2? 2 : 0);
			rn = r.n; rT = r.T; rlen = r.len;
			assigned_any = A1 || A2;
			flippable = r.n >= r.T / 2 + 1;
			for(uint32_t w = 0; w < W; w++)
				has_scg |= scgmask[(uint64_t)s * W + w] != 0;
			if(has_scg && !flippable)                            // can never be assigned to side 1 of a sweep: always counted on side 2
				for(uint32_t w = 0; w < W; w++)
					atomicOr((unsigned long long*)&child_never[((uint64_t)jb.slot * 2 + (sd - 1)) * W + w], (unsigned long long)scgmask[(uint64_t)s * W + w]);
			viol = strategy == ABW_SPLIT_SCAFS && !((double)r.n >= __dmul_rn(fraction_in, (double)r.T));
		}
#pragma unroll
		for(uint32_t sdv = 1; sdv <= 2; sdv++) {
			const bool m = active && sd == sdv;
			const uint32_t ns = __popc(__ballot_sync(0xffffffffu, m));
			if(ns == 0)
				continue;                                        // warp-uniform
			const uint32_t ndps = __reduce_add_sync(0xffffffffu, m? rn : 0u);      // sums stay below 2^31 (N and the sum of T do)
			const uint32_t totT = __reduce_add_sync(0xffffffffu, m? rT : 0u);
			unsigned long long len = m? rlen : 0ull;
#pragma unroll
			for(int o = 16; o > 0; o >>= 1)
				len += __shfl_xor_sync(0xffffffffu, len, o);
			const uint32_t nas = __popc(__ballot_sync(0xffffffffu, m && assigned_any));
			const uint32_t nK = __popc(__ballot_sync(0xffffffffu, m && has_scg && flippable));
			const uint32_t nfl = __popc(__ballot_sync(0xffffffffu, m && flippable));
			const uint32_t nv = __popc(__ballot_sync(0xffffffffu, m && viol));
			if(lane == 0) {
				ChildStats* st = stats + (uint64_t)jb.slot * 2 + (sdv - 1);
				atomicAdd(&st->ndps, (unsigned long long)ndps);
				atomicAdd(&st->totLen, len);
				atomicAdd(&st->ns, ns);
				atomicAdd(&st->totT, totT);
				if(nas) atomicAdd(&st->nassigned, nas);
				if(nK) atomicAdd(&st->K, nK);
				if(nfl) atomicAdd(&st->nflip, nfl);
				if(nv) atomicAdd(&st->viol, nv);
			}
		}
	}
}

// what a level leaves for the next one.  plan_dims[pl]: dimensions of partition plan pl (0: the plan does not exist in this search or at the last level)
__global__ void __launch_bounds__(LV_THREADS) k_level_decide(const LevelBufs B, int cur, int strategy, const abw_params prm, uint32_t Dlocal, uint32_t W,
                                                           uint32_t dim_offset, const uint32_t pd0, const uint32_t pd1, const uint32_t pd2, const uint32_t pd3,
                                                           int build_next, const ChildStats* __restrict__ stats, const unsigned long long* __restrict__ value_key,
                                                           const uint64_t* __restrict__ child_never)
{
	__shared__ uint32_t sm[33];
	__shared__ unsigned long long sm_el;
	LevelCtl* const ctl = B.ctl;
	const LevelCluster* __restrict__ cls = B.cl[cur];
	LevelCluster* __restrict__ nxt = B.cl[cur ^ 1];
	const uint32_t C = ctl->C, nrec0 = ctl->nrec, next_id0 = ctl->next_id, thr = prm.cluster_ndps_threshold, Pmax = B.Pmax;
	if(threadIdx.x == 0)
		sm_el = 0;
	__syncthreads();
	uint32_t P = 0, Tn = 0;
	unsigned long long el = 0;
	for(uint32_t b0 = 0; b0 < C; b0 += LV_THREADS) {
		const uint32_t c = b0 + threadIdx.x;
		const bool valid = c < C;
		bool split = false;
		abw_best br;
		best_reset(br, strategy);
		uint32_t j = 0xFFFFFFFFu;
		if(valid) {
			br = B.bestrec[c];
			j = B.job_of[c];
			if(br.found) {
				const unsigned long long k = value_key[j];
				const unsigned long long bits = (k >> 63)? (k & 0x7FFFFFFFFFFFFFFFull) : ~k;
				br.value = __longlong_as_double((long long)bits);
				if(br.legal) {
					split = !(stats[2 * (size_t)j].ndps < thr || stats[2 * (size_t)j + 1].ndps < thr);      // ClusterSeparator.cpp:125
					if(!split)
						best_reset(br, strategy);                // children too small: best_separation->reset() (:125-132)
				}
			}
		}
		uint32_t tot_s, tot_t;
		const uint32_t exs = cta_excl_scan(split? 1u : 0u, tot_s, sm);
		const uint32_t ext = cta_excl_scan((valid && !split)? 1u : 0u, tot_t, sm);
		if(valid) {
			const LevelCluster lc = cls[c];
			abw_cluster_rec r;
			memset(&r, 0, sizeof(r));
			r.id = lc.id; r.parent = lc.parent; r.ndps = lc.d.n; r.nscafs = lc.nassigned; r.best = br;
			r.gc_avg = r.gc_sd = r.cvg_avg = r.cvg_sd = -1.0;
			if(split) {
				const ChildStats s1 = stats[2 * (size_t)j], s2 = stats[2 * (size_t)j + 1];
				const SplitJob jb = B.jobs[j];
				const uint32_t q = P + exs;
				r.split = 1;
				r.child1 = next_id0 + 2 * q;                     // ids handed out in cluster order, cluster1 first (abawaca.cpp:164-193)
				r.child2 = r.child1 + 1;
				r.child1_ndps = s1.ndps; r.child2_ndps = s2.ndps;
				r.child1_nscafs = s1.nassigned; r.child2_nscafs = s2.nassigned;
				r.child1_raw = jb.swapped? lc.d.n - jb.p : jb.p;
				r.child2_raw = lc.d.n - r.child1_raw;
				uint64_t off = lc.d.off;
				uint32_t kOff = lc.d.kOff, sOff = lc.d.sOff, fOff = lc.d.fOff;
				for(int ch = 0; ch < 2; ch++) {
					const ChildStats& st = ch? s2 : s1;
					LevelCluster hc;
					memset(&hc, 0, sizeof(hc));
					hc.id = ch? r.child2 : r.child1;
					hc.parent = lc.id;
					hc.d.off = off; hc.d.n = (uint32_t)st.ndps;
					hc.d.kOff = kOff; hc.d.K = st.K;
					hc.d.sOff = sOff; hc.d.ns = st.ns;
					hc.d.totT = st.totT; hc.d.U = st.ns; hc.d.totLen = st.totLen;
					hc.d.ss_ok = (st.viol == 0);
					hc.d.fOff = fOff; hc.d.nf = st.nflip;
					hc.nassigned = st.nassigned;
					for(uint32_t w = 0; w < W; w++)
						hc.never[w] = child_never[((size_t)j * 2 + ch) * W + w];
					off += st.ndps; kOff += st.K; sOff += st.ns; fOff += st.nflip;
					nxt[2 * q + ch] = hc;
				}
				PartJob pj;
				pj.off = lc.d.sOff; pj.n = lc.d.ns; pj.n1 = s1.ns;
				B.part_jobs[0 * (size_t)Pmax + q] = pj;
				pj.off = lc.d.off; pj.n = lc.d.n; pj.n1 = (uint32_t)s1.ndps;
				B.part_jobs[1 * (size_t)Pmax + q] = pj;
				pj.off = lc.d.fOff; pj.n = lc.d.nf; pj.n1 = s1.nflip;
				B.part_jobs[2 * (size_t)Pmax + q] = pj;
				pj.off = lc.d.kOff; pj.n = lc.d.K; pj.n1 = s1.K;
				B.part_jobs[3 * (size_t)Pmax + q] = pj;
				if(pd1)
					el += (unsigned long long)lc.d.n * Dlocal;
			}
			else {
				TermJob tj;
				tj.sOff = lc.d.sOff; tj.ns = lc.d.ns; tj.id = lc.id; tj.rec = nrec0 + c;
				B.tjobs[Tn + ext] = tj;
			}
			if(nrec0 + c < B.rec_cap)
				B.recs[nrec0 + c] = r;
		}
		P += tot_s;
		Tn += tot_t;
	}
	__syncthreads();
	const uint32_t Cn = 2 * P;
	// the next level: pass-table offsets, sweep tiles, flip-prefix tiles
	uint32_t tab_total = 0, TT = 0, FPT = 0;
	if(build_next) {
		tab_total = cta_expand(Cn, nullptr, [&](uint32_t i) { return nxt[i].d.K + 1u; }, [&](uint32_t i, uint32_t slot) { nxt[i].d.tabOff = slot; }, sm);
		TT = cta_expand(Cn, B.tile_tab, [&](uint32_t i) { return (nxt[i].d.n + SW_TILE - 1) / SW_TILE; }, [&](uint32_t i, uint32_t slot) { nxt[i].d.tile0 = slot; }, sm);
		if(pd2)
			FPT = cta_expand(Cn, B.fp_tab, [&](uint32_t i) { return (nxt[i].d.nf + FP_TILE - 1) / FP_TILE; }, [](uint32_t, uint32_t) {}, sm);
	}
	// partition plans of this level: scaffold list, elements, flip lists, SCG lists
	const uint32_t pdims[4] = {pd0, pd1, pd2, pd3};
	uint32_t ptt[4], poff[4];
	unsigned long long pend[4];
	uint32_t tab_off = 0;
	unsigned long long item_end = 0;
	for(int pl = 0; pl < 4; pl++) {
		poff[pl] = tab_off;
		ptt[pl] = 0;
		if(pdims[pl]) {
			const PartJob* __restrict__ pj = B.part_jobs + (size_t)pl * Pmax;
			ptt[pl] = cta_expand(P, B.part_tab + tab_off, [&](uint32_t i) { return (pj[i].n + SW_TILE - 1) / SW_TILE; }, [](uint32_t, uint32_t) {}, sm);
		}
		tab_off += ptt[pl];
		item_end += (unsigned long long)ptt[pl] * pdims[pl];
		pend[pl] = item_end;
	}
	// terminal clusters of this level
	const uint32_t tm_items = cta_expand(Tn, B.tm_tab, [&](uint32_t i) { return (B.tjobs[i].ns + TM_CHUNK - 1) / TM_CHUNK; }, [](uint32_t, uint32_t) {}, sm);
	for(uint32_t i = threadIdx.x; i < Tn; i += LV_THREADS) {
		B.tstats[i].total_size = 0;
		B.tstats[i].scg_copies = 0;
	}
	for(uint32_t i = threadIdx.x; i < Tn * W; i += LV_THREADS)
		B.tunion[i] = 0;
	// the one entry of low[] that k_scaf_sides left alone per job
	for(uint32_t k = threadIdx.x; k < ctl->JM; k += LV_THREADS)
		B.low[B.jobs[B.jobs_mine[k]].sstar] = 0;
	atomicAdd(&sm_el, el);
	__syncthreads();
	if(threadIdx.x == 0) {
		ctl->P = P; ctl->Tn = Tn; ctl->TM_items = tm_items; ctl->term_blocks_done = 0;
		for(int pl = 0; pl < 4; pl++) {
			ctl->part_TT[pl] = ptt[pl]; ctl->part_tab_off[pl] = poff[pl]; ctl->part_job_off[pl] = (uint32_t)pl * Pmax; ctl->part_item_end[pl] = pend[pl];
		}
		ctl->partition_elements += sm_el;
		ctl->next_id = next_id0 + 2 * P;
		ctl->nrec = nrec0 + C;
		if(C > 0)                                           // a level the host enqueued past the end of the search is empty and does not count
			ctl->level++;
		ctl->tickets[0] = ctl->tickets[1] = ctl->tickets[2] = 0;
		// the next level (nothing to do in it when no cluster was split)
		ctl->C = build_next? Cn : 0;
		ctl->TT = TT; ctl->FPT = FPT; ctl->tab_total = tab_total;
		ctl->J = ctl->JM = ctl->CL_items = ctl->SS_items = 0;
		ctl->done = (Cn == 0 || ctl->done)? 1u : 0u;
		if(Cn > B.Cmax)
			ctl->error = 2;
		B.prog->c_next[ctl->ticks & 15u] = ctl->C;
		ctl->ticks++;
		if(ctl->done && !ctl->done_at)
			ctl->done_at = ctl->ticks;
		B.prog->error = ctl->error;
		B.prog->done = ctl->done;
		B.prog->done_at = ctl->done_at;
		__threadfence_system();
		B.prog->levels_done = ctl->level;
		B.prog->ticks = ctl->ticks;
		__threadfence_system();
	}
}

// pending clusters become bins without being evaluated (abw_search_set_max_levels): the children of the last level that was run
__global__ void __launch_bounds__(LV_THREADS) k_pending_jobs(const LevelBufs B, int cur, uint32_t W)
{
	__shared__ uint32_t sm[33];
	LevelCtl* const ctl = B.ctl;
	const LevelCluster* __restrict__ cls = B.cl[cur];
	const uint32_t Tn = 2 * ctl->P;
	for(uint32_t i = threadIdx.x; i < Tn; i += LV_THREADS) {
		TermJob tj;
		tj.sOff = cls[i].d.sOff; tj.ns = cls[i].d.ns; tj.id = cls[i].id; tj.rec = 0xFFFFFFFFu;
		B.tjobs[i] = tj;
		B.tstats[i].total_size = 0;
		B.tstats[i].scg_copies = 0;
	}
	for(uint32_t i = threadIdx.x; i < Tn * W; i += LV_THREADS)
		B.tunion[i] = 0;
	__syncthreads();
	const uint32_t tm_items = cta_expand(Tn, B.tm_tab, [&](uint32_t i) { return (B.tjobs[i].ns + TM_CHUNK - 1) / TM_CHUNK; }, [](uint32_t, uint32_t) {}, sm);
	if(threadIdx.x == 0) {
		ctl->Tn = Tn; ctl->TM_items = tm_items; ctl->term_blocks_done = 0;
	}
}

// terminal cluster: bins of its scaffolds and datapoints (abawaca.cpp:135-138), total size and SCG tallies (ClusterQuality.cpp:44-48,78-87).  The last CTA to
// finish completes the records: SCGdb::num_unique_scgs / average_num_copies_for_unique_scgs (SCGdb.cpp:6-18,41-55) and, when per-scaffold G+C and coverage were
// given, the summary statistics of the bin (ClusterQuality::gc / cvg with standard_deviation, ClusterQuality.cpp:6-27,51-75): over the ASSIGNED scaffolds of the
// bin in scaffold-id order (std::set iteration), mean = sum(len * x) / sum(len), stdev = sqrt(sum(len * (x - mean) * (x - mean)) / (sum(len) - 1)), evaluated
// with exactly those fp64 operations in that order; (-1, -1) for a bin without assigned scaffolds.  The scaffold list of a cluster stays in ascending id order
// through the stable partitions, so one thread walks its bin.
__global__ void __launch_bounds__(128) k_finalize_terminal(const uint32_t* __restrict__ scaf_list, const LevelBufs B, const ScafRow* __restrict__ rows,
                                    const uint8_t* __restrict__ assigned, const uint64_t* __restrict__ scgmask, uint32_t W, uint32_t* __restrict__ scaf_member,
                                    uint32_t* __restrict__ scaf_final, const double* __restrict__ x_gc, const double* __restrict__ x_cvg)
{
	__shared__ int sm_last;
	LevelCtl* const ctl = B.ctl;
	const uint32_t items = ctl->TM_items, Tn = ctl->Tn;
	for(uint32_t it = blockIdx.x; it < items; it += gridDim.x) {
		const uint2 te = B.tm_tab[it];
		const TermJob jb = B.tjobs[te.x];
		const uint32_t i1 = min(jb.ns, (te.y + 1) * TM_CHUNK);
		for(uint32_t i = te.y * TM_CHUNK + threadIdx.x; i < i1; i += blockDim.x) {
			const uint32_t s = scaf_list[jb.sOff + i] & EL_SCAF_MASK;
			scaf_member[s] = jb.id;
			if(assigned[s]) {
				scaf_final[s] = jb.id;
				atomicAdd(&B.tstats[te.x].total_size, (unsigned long long)rows[s].len);
				uint32_t copies = 0;
				for(uint32_t w = 0; w < W; w++) {
					const uint64_t m = scgmask[(uint64_t)s * W + w];
					if(m) {
						copies += __popcll(m);
						atomicOr((unsigned long long*)&B.tunion[(uint64_t)te.x * W + w], (unsigned long long)m);
					}
				}
				if(copies)
					atomicAdd(&B.tstats[te.x].scg_copies, (unsigned long long)copies);
			}
		}
	}
	__threadfence();
	__syncthreads();
	if(threadIdx.x == 0)
		sm_last = (atomicAdd(&ctl->term_blocks_done, 1u) == gridDim.x - 1);
	__syncthreads();
	if(!sm_last)
		return;
	__threadfence();
	for(uint32_t q = threadIdx.x; q < Tn; q += blockDim.x) {
		const TermJob jb = B.tjobs[q];
		if(jb.rec >= B.rec_cap)
			continue;
		uint32_t u = 0;
		for(uint32_t w = 0; w < W; w++)
			u += (uint32_t)__popcll(__ldcg((const unsigned long long*)&B.tunion[(uint64_t)q * W + w]));
		const unsigned long long size = __ldcg(&B.tstats[q].total_size), copies = __ldcg(&B.tstats[q].scg_copies);
		abw_cluster_rec* r = B.recs + jb.rec;
		r->total_size = size;
		r->scg_unique = u;
		r->scg_avg = (copies == 0)? 0.0 : __ddiv_rn((double)copies, (double)u);   // SCGdb.cpp:54
	}
	if(x_gc != nullptr) {
		for(uint32_t t = threadIdx.x; t < 2 * Tn; t += blockDim.x) {
			const TermJob jb = B.tjobs[t >> 1];
			if(jb.rec >= B.rec_cap)
				continue;
			const double* __restrict__ x = (t & 1)? x_cvg : x_gc;
			unsigned long long total = 0;
			uint32_t count = 0;
			double mean = 0.0;
			for(uint32_t i = 0; i < jb.ns; i++) {
				const uint32_t sc = scaf_list[jb.sOff + i] & EL_SCAF_MASK;
				if(assigned[sc]) {
					const unsigned long long l = rows[sc].len;
					mean = __dadd_rn(mean, __dmul_rn(__ull2double_rn(l), x[sc]));
					total += l;
					count++;
				}
			}
			double sd = 0.0;
			if(count == 0)
				mean = sd = -1.0;
			else {
				mean = __ddiv_rn(mean, __ull2double_rn(total));
				for(uint32_t i = 0; i < jb.ns; i++) {
					const uint32_t sc = scaf_list[jb.sOff + i] & EL_SCAF_MASK;
					if(assigned[sc]) {
						const double dlt = __dsub_rn(x[sc], mean);
						sd = __dadd_rn(sd, __dmul_rn(__dmul_rn(__ull2double_rn(rows[sc].len), dlt), dlt));
					}
				}
				sd = __dsqrt_rn(__ddiv_rn(sd, __ull2double_rn(total - 1ull)));
			}
			abw_cluster_rec* r = B.recs + jb.rec;
			if(t & 1) { r->cvg_avg = mean; r->cvg_sd = sd; }
			else { r->gc_avg = mean; r->gc_sd = sd; }
		}
	}
}

// ---------------------------------------------------------------------------------------------------
// stable partition of the elements of the split clusters, every dimension (same warp-striped rows as k_sweep_ss); the boundary flag of an
// element becomes "value differs from the previous element OF ITS NEW CLUSTER", i.e. the OR of the flags since that element.  Lane r owns the masks of row r:
//   S1 = elements that go to child 1, S2 = to child 2, B = boundary flags.
// New flag of an element of child X = OR of the old flags since the previous element of child X (itself included).  With the closers
// P = SX that is a carry chain:  (B & ~P) + ~P  overflows a run of non-closers exactly when the run holds a boundary, and the carry
// lands on the closer that ends the run.  A run of elements is summarised per child by H ("contains an element of the child") and
// T ("a boundary is pending after the last such element"); summaries compose associatively, so rows, warps and tiles chain with a
// scan and the usual look-back.  The scaffold list, the flip lists and the SCG lists of the level are u32 lists partitioned by the same launch
// ("plans": work items of all plans share one ticket); the scaffold-list plan also commits the new assignment of every scaffold it moves.
// ---------------------------------------------------------------------------------------------------
// bits: 0 = H1, 1 = H2, 2 = T1, 3 = T2
__device__ __forceinline__ uint32_t ht_compose(uint32_t first, uint32_t then)
{
	const uint32_t H = (first | then) & 3u;
	const uint32_t T = ((then >> 2) | ((first >> 2) & ~then)) & 3u;
	return H | (T << 2);
}
// pending state (bit 0: child 1, bit 1: child 2) after a run with summary ht entered in `state`
__device__ __forceinline__ uint32_t ht_apply(uint32_t ht, uint32_t state) { return ((ht >> 2) | (state & ~ht)) & 3u; }

// payload of the partition's packed look-back word (lb_pack): count of child-1 elements, summary bits (an inclusive prefix has the pending state there)
__device__ __forceinline__ unsigned long long lb2_payload(uint32_t cnt, uint32_t ht) { return (unsigned long long)cnt | ((unsigned long long)ht << 32); }

struct PartPlans {
	const uint32_t* in[4];
	uint32_t*       out[4];
	uint64_t        stride[4];
};

__global__ void __launch_bounds__(SW_THREADS, PART_CTAS) k_partition2(const PartPlans plans, LevelCtl* __restrict__ ctl, const PartJob* __restrict__ jobs_all,
                                                             const uint2* __restrict__ tab_all, const uint8_t* __restrict__ side, const uint8_t* __restrict__ new_assigned,
                                                             uint8_t* __restrict__ assigned, uint32_t epoch, unsigned long long* __restrict__ lookback)
{
	__shared__ uint32_t sm_cnt[SW_THREADS / 32];
	__shared__ uint32_t sm_ht[SW_THREADS / 32];
	__shared__ unsigned long long sm_w;
	const unsigned long long end0 = ctl->part_item_end[0], end1 = ctl->part_item_end[1], end2 = ctl->part_item_end[2], end3 = ctl->part_item_end[3];
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	while(true) {
		if(threadIdx.x == 0)
			sm_w = atomicAdd(&ctl->tickets[2], 1ull);
		__syncthreads();
		const uint64_t w = sm_w;
		if(w >= end3)
			break;
		const int pl = (w >= end0) + (w >= end1) + (w >= end2);
		const uint64_t wl = w - ((pl == 0)? 0ull : (pl == 1)? end0 : (pl == 2)? end1 : end2);
		const uint32_t TT = ctl->part_TT[pl];
		const uint32_t d = (uint32_t)(wl / TT);
		const uint2 te = __ldg(tab_all + ctl->part_tab_off[pl] + (uint32_t)(wl - (uint64_t)d * TT));
		const PartJob jb = jobs_all[ctl->part_job_off[pl] + te.x];
		const uint32_t tile = te.y;
		const uint64_t stride = plans.stride[pl];
		const uint32_t* __restrict__ src = plans.in[pl] + (uint64_t)d * stride + jb.off;
		uint32_t* __restrict__ dst1 = plans.out[pl] + (uint64_t)d * stride + jb.off;
		uint32_t* __restrict__ dst2 = dst1 + jb.n1;
		const uint32_t wbase = tile * SW_TILE + warp * SW_WARP_CHUNK;
		uint32_t el[32];
		uint32_t my1 = 0;                                      // bit r: my element of row r goes to child 1
		uint32_t mS1 = 0, mV = 0, mB = 0;                      // masks of row `lane`
		const bool active = wbase < jb.n;
		const bool full = wbase + SW_WARP_CHUNK <= jb.n;       // warp uniform: all 1024 elements of the chunk exist, no bounds checks
		if(full) {
#pragma unroll
			for(int r = 0; r < 32; r++)
				el[r] = __ldg(src + wbase + r * 32 + lane);
			mV = 0xFFFFFFFFu;
#pragma unroll
			for(int r = 0; r < 32; r++) {
				const bool is1 = side[el[r] & EL_SCAF_MASK] == 1;
				const uint32_t s1 = __ballot_sync(0xffffffffu, is1);
				const uint32_t b = __ballot_sync(0xffffffffu, el[r] >> 31);
				my1 |= (is1? 1u : 0u) << r;
				if(lane == r) { mS1 = s1; mB = b; }
			}
		}
		else if(active) {
#pragma unroll
			for(int r = 0; r < 32; r++) {
				const uint32_t idx = wbase + r * 32 + lane;
				el[r] = (idx < jb.n)? __ldg(src + idx) : 0xFFFFFFFFu;
			}
#pragma unroll
			for(int r = 0; r < 32; r++) {
				const uint32_t idx = wbase + r * 32 + lane;
				const bool valid = idx < jb.n;
				const bool is1 = valid && side[el[r] & EL_SCAF_MASK] == 1;
				const uint32_t s1 = __ballot_sync(0xffffffffu, is1);
				const uint32_t v = __ballot_sync(0xffffffffu, valid);
				const uint32_t b = __ballot_sync(0xffffffffu, valid && (el[r] >> 31));
				my1 |= (is1? 1u : 0u) << r;
				if(lane == r) { mS1 = s1; mV = v; mB = b; }
			}
		}
		const uint32_t mS2 = mV & ~mS1;
		const uint32_t c1 = __popc(mS1);
		const unsigned long long s1sum = (unsigned long long)(mB & ~mS1) + (unsigned long long)(uint32_t)(~mS1);
		const unsigned long long s2sum = (unsigned long long)(mB & ~mS2) + (unsigned long long)(uint32_t)(~mS2);
		uint32_t newflags = (((uint32_t)s1sum | mB) & mS1) | (((uint32_t)s2sum | mB) & mS2);     // assuming nothing is pending when the row starts
		const uint32_t myht = (mS1? 1u : 0u) | (mS2? 2u : 0u) | ((uint32_t)(s1sum >> 32) << 2) | ((uint32_t)(s2sum >> 32) << 3);
		// inclusive scans over the rows of the warp
		uint32_t icnt = c1, iht = myht;
#pragma unroll
		for(int o = 1; o < 32; o <<= 1) {
			const uint32_t c2 = __shfl_up_sync(0xffffffffu, icnt, o), h2 = __shfl_up_sync(0xffffffffu, iht, o);
			if(lane >= o) {
				icnt += c2;
				iht = ht_compose(h2, iht);
			}
		}
		if(lane == 31) {
			sm_cnt[warp] = icnt;
			sm_ht[warp] = iht;
		}
		__syncthreads();
		if(threadIdx.x < 32) {
			// exclusive over the warps (every lane computes the same), then the look-back over the earlier tiles of this (job, dimension)
			uint32_t rc = 0, rh = 0;
			uint32_t wc = 0, wh = 0;
#pragma unroll
			for(int w2 = 0; w2 < SW_THREADS / 32; w2++) {
				const uint32_t tc = sm_cnt[w2], th = sm_ht[w2];
				if(w2 == lane) { wc = rc; wh = rh; }
				rc += tc;
				rh = ht_compose(rh, th);
			}
			uint32_t carry_cnt = 0, carry_state = 3u;          // the first element of each child gets its boundary flag set
			if(tile > 0) {
				if(lane == 0)
					st_volatile_u64(&lookback[w], lb_pack(lb2_payload(rc, rh), LB_AGG, epoch));
				uint32_t acc = 0;                               // summary of the tiles between the window and this tile
				const bool ok = lb_walk(w, tile, [&](uint64_t i) { return ld_volatile_u64(&lookback[i]); },
				                        [&](unsigned long long v) { return lb_packed_state(v, epoch); },
				                        [&](unsigned long long v, uint64_t, bool take, uint32_t first_prefix) {
					carry_cnt += __reduce_add_sync(0xffffffffu, take? (uint32_t)v : 0u);
					// summaries compose in tile order and higher lanes are EARLIER tiles: suffix-compose towards lane 0
					uint32_t h = (take && (uint32_t)lane != first_prefix)? ((uint32_t)(v >> 32) & 0xFu) : 0u;      // identity for lanes that do not take part
#pragma unroll
					for(int o = 1; o < 32; o <<= 1) {
						const uint32_t hh = __shfl_down_sync(0xffffffffu, h, o);
						if(lane + o < 32)
							h = ht_compose(hh, h);
					}
					const uint32_t window = __shfl_sync(0xffffffffu, h, 0);            // all aggregates of the window, earliest first
					if(first_prefix < 32u) {
						const uint32_t state_at_prefix = (uint32_t)(__shfl_sync(0xffffffffu, v, (int)first_prefix) >> 32) & 3u;
						carry_state = ht_apply(acc, ht_apply(window, state_at_prefix));
					}
					else
						acc = ht_compose(window, acc);
				});
				if(!ok && lane == 0)
					atomicExch(&ctl->error, 1u);
			}
			if(lane == 0)
				st_volatile_u64(&lookback[w], lb_pack(lb2_payload(carry_cnt + rc, ht_apply(rh, carry_state)), LB_PREFIX, epoch));
			if(lane < SW_THREADS / 32) {
				sm_cnt[lane] = carry_cnt + wc;                  // child-1 elements before warp `lane`
				sm_ht[lane] = ht_apply(wh, carry_state);        // pending state when warp `lane` starts
			}
		}
		__syncthreads();
		if(active) {
			uint32_t ecnt = __shfl_up_sync(0xffffffffu, icnt, 1), eht = __shfl_up_sync(0xffffffffu, iht, 1);
			if(lane == 0) {
				ecnt = 0;
				eht = 0;
			}
			const uint32_t row_before1 = sm_cnt[warp] + ecnt;
			const uint32_t state = ht_apply(eht, sm_ht[warp]);      // pending when my row starts: lands on the first element of each child in the row
			if(state & 1u)
				newflags |= mS1 & (0u - mS1);
			if(state & 2u)
				newflags |= mS2 & (0u - mS2);
			const uint32_t lt = (1u << lane) - 1u;
			const bool commit = (pl == 0);                      // the scaffold list: every scaffold of a split cluster passes here exactly once
			if(full) {
#pragma unroll
				for(int r = 0; r < 32; r++) {
					const uint32_t S1r = __shfl_sync(0xffffffffu, mS1, r), Fr = __shfl_sync(0xffffffffu, newflags, r), b1 = __shfl_sync(0xffffffffu, row_before1, r);
					const uint32_t idx = wbase + r * 32 + lane;
					const uint32_t before1 = b1 + __popc(S1r & lt);
					const uint32_t e = (el[r] & 0x7FFFFFFFu) | (((Fr >> lane) & 1u) << 31);
					uint32_t* const dst = ((my1 >> r) & 1u)? dst1 + before1 : dst2 + (idx - before1);
					*dst = e;
					if(commit)
						assigned[el[r] & EL_SCAF_MASK] = new_assigned[el[r] & EL_SCAF_MASK] != 0;
				}
			}
			else {
#pragma unroll
				for(int r = 0; r < 32; r++) {
					const uint32_t S1r = __shfl_sync(0xffffffffu, mS1, r), Fr = __shfl_sync(0xffffffffu, newflags, r), b1 = __shfl_sync(0xffffffffu, row_before1, r);
					const uint32_t idx = wbase + r * 32 + lane;
					if(idx < jb.n) {
						const uint32_t before1 = b1 + __popc(S1r & lt);
						const uint32_t e = (el[r] & 0x7FFFFFFFu) | (((Fr >> lane) & 1u) << 31);
						if((my1 >> r) & 1u)
							dst1[before1] = e;
						else
							dst2[idx - before1] = e;
						if(commit)
							assigned[el[r] & EL_SCAF_MASK] = new_assigned[el[r] & EL_SCAF_MASK] != 0;
					}
				}
			}
		}
		__syncthreads();
	}
}

// ClusterQuality::scg for an arbitrary scaffold list (abw_cluster_scg): OR and copy count of the SCG sets
__global__ void k_scg_tally(const uint32_t* __restrict__ list, uint32_t n, const uint64_t* __restrict__ scgmask, uint32_t W, TermStats* __restrict__ stats,
                            uint64_t* __restrict__ union_mask)
{
	for(uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
		const uint32_t s = list[i];
		uint32_t copies = 0;
		for(uint32_t w = 0; w < W; w++) {
			const uint64_t m = scgmask[(uint64_t)s * W + w];
			if(m) {
				copies += __popcll(m);
				atomicOr((unsigned long long*)&union_mask[w], (unsigned long long)m);
			}
		}
		if(copies)
			atomicAdd(&stats->scg_copies, (unsigned long long)copies);
	}
}

__global__ void k_dp_bins(const uint32_t* __restrict__ dp2scaf, const uint32_t* __restrict__ scaf_member, uint64_t N, uint32_t* __restrict__ dp2cluster)
{
	uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if(i < N)
		dp2cluster[i] = scaf_member[dp2scaf[i]];
}

// ---------------------------------------------------------------------------------------------------
// build: keys, within-scaffold classes, element packing
// ---------------------------------------------------------------------------------------------------
// Sort keys of the dimensions [d0, d0 + nd) of all datapoints, column major [nd][N], and the datapoint index beside each.
// MILLI: columns written by abawaca-build hold multiples of 0.001 (int(1000*x)/1000.0, abawaca-build.cpp:603).  When every value v satisfies
// v == (double)k / 1000.0 for the integer k = rint(1000*v), |k| < 2^31, ordering by k is ordering by v (ties included) and the sort runs on 32-bit keys
// with few significant bits; any other value sets flag[0] and the chunk is redone with the 64-bit keys (an order-preserving image of the double; -0.0 and
// +0.0 compare equal in comp_by_value, ClusterSeparator.cpp:8; NaN sets flag[1]).
// One CTA transposes a tile of 32 datapoints x 32 dimensions through shared memory: coalesced reads of a row-major matrix, coalesced writes of the keys.
template <bool MILLI, typename KeyT>
__global__ void __launch_bounds__(256) k_keys(const ValSrc v, uint64_t N, uint32_t d0, uint32_t nd, KeyT* __restrict__ keys, uint32_t* __restrict__ vals,
                                              int* __restrict__ flag)
{
	__shared__ KeyT tile[32][33];
	const uint64_t r0 = (uint64_t)blockIdx.x * 32;
	const uint32_t c0 = blockIdx.y * 32;
	const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
	bool bad = false, isnan = false;
	const bool rowmajor = v.layout != ABW_LAYOUT_COLMAJOR;
#pragma unroll
	for(int j = 0; j < 4; j++) {
		// row-major: x runs over the dimensions of one datapoint; column-major: x runs over the datapoints of one dimension
		const uint64_t dp = rowmajor? r0 + ty + 8 * j : r0 + tx;
		const uint32_t c = rowmajor? c0 + tx : c0 + ty + 8 * j;
		KeyT key = 0;
		if(dp < N && c < nd) {
			if(MILLI && v.layout == ABW_LAYOUT_ROWMAJOR_MILLI32) {
				// the matrix already holds the integers
				const uint32_t u = reinterpret_cast<const uint32_t*>(v.p)[(v.rowidx? v.rowidx[dp] : dp) * v.ld + d0 + c];
				bad |= u >= 2147483000u;
				key = (KeyT)(u + 2147483648u);
			}
			else {
				const double x = val_at(v, dp, d0 + c);
				if(MILLI) {
					const double k = rint(__dmul_rn(x, 1000.0));
					const bool ok = (k > -2147483000.0) && (k < 2147483000.0) && (__ddiv_rn(k, 1000.0) == x);
					bad |= !ok;
					key = (KeyT)(ok? (uint32_t)((long long)k + 2147483648ll) : 0u);
				}
				else {
					isnan |= x != x;
					key = (KeyT)orderable(x);
				}
			}
		}
		if(rowmajor)
			tile[ty + 8 * j][tx] = key;                     // [datapoint][dimension]
		else
			tile[tx][ty + 8 * j] = key;
	}
	__syncthreads();
#pragma unroll
	for(int j = 0; j < 4; j++) {
		const uint32_t c = c0 + ty + 8 * j;
		const uint64_t dp = r0 + tx;
		if(dp < N && c < nd) {
			keys[(uint64_t)c * N + dp] = tile[tx][ty + 8 * j];
			vals[(uint64_t)c * N + dp] = (uint32_t)dp;
		}
	}
	if(__syncthreads_or(bad || isnan)) {
		if(bad)
			atomicExch(&flag[0], 1);
		if(isnan)
			atomicExch(&flag[1], 1);
	}
}

__global__ void k_fill_or_and(uint32_t* __restrict__ or_and, uint32_t n)
{
	const uint32_t d = blockIdx.x * blockDim.x + threadIdx.x;
	if(d < n) {
		or_and[2 * d] = 0u;
		or_and[2 * d + 1] = ~0u;
	}
}

// class of every datapoint in every dimension of the chunk, from its rank inside its scaffold (ties by datapoint index,
// the order a stable sort produces).  Thread per (datapoint, dimension), on the sort keys (same order as the values, ties included).
template <typename KeyT>
__global__ void __launch_bounds__(256) k_rank_class(const KeyT* __restrict__ keys, uint64_t N, uint32_t nd, const uint32_t* __restrict__ dp2scaf,
                                                    const uint64_t* __restrict__ dp_first, const ScafRow* __restrict__ rows, const uint8_t* __restrict__ has_scg, int strategy,
                                                    double fraction_in, uint8_t* __restrict__ cls_out, uint32_t* __restrict__ or_and)
{
	const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
	const uint32_t d = blockIdx.y;
	if(or_and != nullptr) {
		// OR and AND of the (32-bit) keys of dimension d (or_and[2 d], or_and[2 d + 1], preset to 0 and ~0): which key bits differ at all, per dimension --
		// k-mer thousandths fit one radix digit, coverage needs two.  One atomic pair per CTA.
		__shared__ uint32_t sm_or[8], sm_and[8];
		const uint32_t k32 = (i < N && d < nd)? (uint32_t)keys[(uint64_t)d * N + i] : 0u;
		const uint32_t o = __reduce_or_sync(0xffffffffu, k32), a = __reduce_and_sync(0xffffffffu, (i < N && d < nd)? k32 : ~0u);
		if((threadIdx.x & 31) == 0) {
			sm_or[threadIdx.x >> 5] = o;
			sm_and[threadIdx.x >> 5] = a;
		}
		__syncthreads();
		if(threadIdx.x == 0 && d < nd) {
			uint32_t oo = 0u, aa = ~0u;
#pragma unroll
			for(int w = 0; w < 8; w++) {
				oo |= sm_or[w];
				aa &= sm_and[w];
			}
			atomicOr(&or_and[2 * d], oo);
			atomicAnd(&or_and[2 * d + 1], aa);
		}
	}
	if(i >= N || d >= nd)
		return;
	const uint32_t s = dp2scaf[i];
	const ScafRow r = rows[s];
	const uint64_t f = dp_first[s];
	const KeyT* __restrict__ col = keys + (uint64_t)d * N;
	const KeyT ki = col[i];
	uint32_t a = 1;                                              // 1-based rank of this dp among the dps of its scaffold
	for(uint64_t j = f; j < f + r.n; j++) {
		const KeyT kj = __ldg(col + j);
		a += (kj < ki) || (kj == ki && j < i);
	}
	uint32_t cls, aux;
	if(strategy == ABW_SENS_SPEC) {
		const uint32_t flip = r.T / 2 + 1;                       // first a with 2*a > T (...Specificity.cpp:125)
		cls = (a < flip)? 0u : (a == flip)? 1u : 2u;
		aux = (a == flip && has_scg[s])? 1u : 0u;
	}
	else {
		const uint32_t r1 = (uint32_t)ceil(__dmul_rn(fraction_in, (double)r.T));   // first a with a >= fraction*T (...SplitScafs.h:85-86)
		const uint32_t r2 = r.n - r1 + 1;                                             // the a whose removal drops side 2 below fraction*T
		cls = (a < r1)? 0u : (a == r1)? 1u : 2u;
		aux = (r1 > r.n)? 2u : ((a < r2)? 0u : (a == r2)? 1u : 2u);                   // r1 > n: the scaffold is never "in" either side
	}
	cls_out[(uint64_t)d * N + i] = (uint8_t)(cls | (aux << 2));
}

template <typename KeyT>
__global__ void k_pack_elements(const KeyT* __restrict__ keys, const uint32_t* __restrict__ vals, uint64_t N, uint32_t nd, const uint32_t* __restrict__ dp2scaf,
                                const uint8_t* __restrict__ cls, uint32_t* __restrict__ E, const uint32_t* __restrict__ scg_index, uint32_t* __restrict__ flip_pos, uint64_t K)
{
	const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
	const uint32_t d = blockIdx.y;
	if(i >= N || d >= nd)
		return;
	const uint64_t o = (uint64_t)d * N + i;
	const uint32_t dp = vals[o];
	const uint32_t s = dp2scaf[dp];
	const uint32_t c = cls[(uint64_t)d * N + dp];
	const uint32_t boundary = (i == 0) || (keys[o] != keys[o - 1]);
	E[o] = s | ((c & 3u) << EL_CLASS_SHIFT) | (((c >> 2) & 3u) << EL_AUX_SHIFT) | (boundary? EL_BOUNDARY : 0u);
	if(flip_pos != nullptr && (c & 3u) == 1u && ((c >> 2) & 1u))
		flip_pos[(uint64_t)d * K + scg_index[s]] = (uint32_t)i;
}

// ---------------------------------------------------------------------------------------------------
// per-scaffold tables of a problem, built on the device from the caller's arrays (dp2scaf, T, len, scgmask)
// ---------------------------------------------------------------------------------------------------
constexpr int TB_ERR_RANGE = 1, TB_ERR_ORDER = 2, TB_ERR_COUNT = 4, TB_ERR_T = 8;
struct RootStats {
	unsigned long long totT, totLen;
	uint32_t viol, Sf, partial, err;
	unsigned long long never[SCG_WMAX];
};

// one thread per datapoint: dp2scaf must be non-decreasing, below S and without gaps; first[s] = first datapoint of scaffold s
__global__ void k_tab_runs(const uint32_t* __restrict__ dp2scaf, uint64_t N, uint32_t S, uint64_t* __restrict__ first, RootStats* __restrict__ rs)
{
	const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if(i >= N)
		return;
	const uint32_t sc = dp2scaf[i];
	int err = 0;
	if(sc >= S)
		err |= TB_ERR_RANGE;
	else if(i == 0) {
		if(sc != 0)
			err |= TB_ERR_COUNT;                            // scaffold 0 has no datapoint
		first[0] = 0;
	}
	else {
		const uint32_t prev = dp2scaf[i - 1];
		if(prev > sc)
			err |= TB_ERR_ORDER;
		else if(prev != sc) {
			if(sc - prev > 1)
				err |= TB_ERR_COUNT;                        // a scaffold in between has no datapoint
			first[sc] = i;
		}
	}
	if(i == N - 1) {
		if(sc < S && sc != S - 1)
			err |= TB_ERR_COUNT;
		first[S] = N;
	}
	if(err)
		atomicOr(&rs->err, (uint32_t)err);
}

// dp2scaf of a matrix that holds every datapoint of every scaffold (n == T, the reference's own flow): datapoints [first[s], first[s+1]) belong to s
__global__ void k_tab_fill_dp2scaf(const uint64_t* __restrict__ first, uint32_t S, uint64_t N, uint32_t* __restrict__ dp2scaf)
{
	const uint32_t sidx = blockIdx.x * blockDim.x + threadIdx.x;
	if(sidx >= S)
		return;
	const uint64_t a = first[sidx], b = min(first[sidx + 1], N);
	for(uint64_t i = a; i < b; i++)
		dp2scaf[i] = sidx;
}

// one thread per scaffold: {T, n, len} row, SCG flag, root statistics (warp-aggregated)
__global__ void __launch_bounds__(256) k_tab_scaffolds(const uint64_t* __restrict__ first, const uint32_t* __restrict__ T, const uint64_t* __restrict__ len,
                                                       const uint64_t* __restrict__ scgmask, uint32_t S, uint32_t W, double fraction_in, ScafRow* __restrict__ rows,
                                                       uint4* __restrict__ frow, uint8_t* __restrict__ has_scg, uint32_t* __restrict__ scg_flag, uint32_t* __restrict__ scaf_iota, RootStats* __restrict__ rs)
{
	const uint32_t sidx = blockIdx.x * blockDim.x + threadIdx.x;
	const bool active = sidx < S;
	uint32_t t = 0, n = 0, err = 0;
	unsigned long long l = 0;
	bool any = false, flippable = false, viol = false, partial = false;
	if(active) {
		t = T[sidx];
		l = len[sidx];
		const uint64_t n64 = first[sidx + 1] - first[sidx];
		n = (uint32_t)min(n64, (uint64_t)0xFFFFFFFFu);
		if(t < 2)
			err |= TB_ERR_T;
		if(n == 0 || n > t)
			err |= TB_ERR_COUNT;
		for(uint32_t w = 0; w < W; w++)
			any |= scgmask[(uint64_t)sidx * W + w] != 0;
		flippable = n >= t / 2 + 1;
		viol = !((double)n >= fraction_in * (double)t);
		partial = n != t;
		ScafRow r;
		r.T = t; r.n = n; r.len = l;
		rows[sidx] = r;
		frow[sidx] = make_uint4(t, n | ((any? 1u : 0u) << 31), (uint32_t)l, (uint32_t)(l >> 32));     // the same with the SCG flag inside: one gather per flip-list entry
		has_scg[sidx] = any;
		scg_flag[sidx] = (any && flippable)? 1u : 0u;
		scaf_iota[sidx] = sidx;
		if(any && !flippable)                               // can never be assigned to side 1 of a sweep: always counted on side 2
			for(uint32_t w = 0; w < W; w++)
				atomicOr(&rs->never[w], (unsigned long long)scgmask[(uint64_t)sidx * W + w]);
	}
	unsigned long long st = t, sl = l;
#pragma unroll
	for(int o = 16; o > 0; o >>= 1) {
		st += __shfl_xor_sync(0xffffffffu, st, o);
		sl += __shfl_xor_sync(0xffffffffu, sl, o);
	}
	const uint32_t nv = __popc(__ballot_sync(0xffffffffu, active && viol)), nf = __popc(__ballot_sync(0xffffffffu, active && flippable)),
	               np = __popc(__ballot_sync(0xffffffffu, active && partial));
	err = __reduce_or_sync(0xffffffffu, err);
	if((threadIdx.x & 31) == 0) {
		atomicAdd(&rs->totT, st);
		atomicAdd(&rs->totLen, sl);
		if(nv) atomicAdd(&rs->viol, nv);
		if(nf) atomicAdd(&rs->Sf, nf);
		if(np) atomicAdd(&rs->partial, np);
		if(err) atomicOr(&rs->err, err);
	}
}

// SCG-carrying scaffolds that can flip, in scaffold order, and the index of each in that list
__global__ void k_tab_scg(const uint32_t* __restrict__ scg_flag, const uint64_t* __restrict__ scg_before, uint32_t S, uint32_t* __restrict__ scg_index, uint32_t* __restrict__ scg_scafs)
{
	const uint32_t sidx = blockIdx.x * blockDim.x + threadIdx.x;
	if(sidx >= S)
		return;
	const uint32_t k = (uint32_t)scg_before[sidx];
	scg_index[sidx] = scg_flag[sidx]? k : 0u;
	if(scg_flag[sidx])
		scg_scafs[k] = sidx;
}

// flip list of every dimension: the scaffold ids of the class-1 elements in element order (stream compaction of E).
// pass 1: class-1 elements per tile of SW_TILE; pass 2: a tile finds its offset by summing the counts of the tiles before it.
__global__ void __launch_bounds__(256) k_flip_count(const uint32_t* __restrict__ E, uint64_t N, uint32_t tiles, uint32_t* __restrict__ counts)
{
	__shared__ uint32_t sm[8];
	const uint32_t d = blockIdx.y, t = blockIdx.x;
	const uint32_t* __restrict__ seg = E + (uint64_t)d * N;
	const uint64_t i1 = min(N, (uint64_t)(t + 1) * SW_TILE);
	uint32_t c = 0;
	for(uint64_t i = (uint64_t)t * SW_TILE + threadIdx.x; i < i1; i += 256)
		c += (seg[i] >> EL_CLASS_SHIFT) & 1u;
	c = __reduce_add_sync(0xffffffffu, c);
	if((threadIdx.x & 31) == 0)
		sm[threadIdx.x >> 5] = c;
	__syncthreads();
	if(threadIdx.x == 0)
		counts[(uint64_t)d * tiles + t] = sm[0] + sm[1] + sm[2] + sm[3] + sm[4] + sm[5] + sm[6] + sm[7];
}

__global__ void __launch_bounds__(256) k_flip_write(const uint32_t* __restrict__ E, uint64_t N, uint32_t tiles, const uint32_t* __restrict__ counts, uint32_t* __restrict__ list,
                                                   uint64_t Sf)
{
	__shared__ uint32_t sm[9];
	const uint32_t d = blockIdx.y, t = blockIdx.x;
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	uint32_t before = 0;
	for(uint32_t i = threadIdx.x; i < t; i += 256)
		before += counts[(uint64_t)d * tiles + i];
	before = __reduce_add_sync(0xffffffffu, before);
	if(lane == 0)
		sm[warp] = before;
	__syncthreads();
	uint32_t run = sm[0] + sm[1] + sm[2] + sm[3] + sm[4] + sm[5] + sm[6] + sm[7];
	__syncthreads();
	const uint32_t* __restrict__ seg = E + (uint64_t)d * N;
	uint32_t* __restrict__ out = list + (uint64_t)d * Sf;
	const uint64_t i0 = (uint64_t)t * SW_TILE, i1 = min(N, i0 + SW_TILE);
	for(uint64_t base = i0; base < i1; base += 256) {
		const uint64_t i = base + threadIdx.x;
		const uint32_t e = (i < i1)? seg[i] : 0u;
		const bool flip = (e >> EL_CLASS_SHIFT) & 1u;
		const uint32_t bal = __ballot_sync(0xffffffffu, flip);
		if(lane == 0)
			sm[warp] = __popc(bal);
		__syncthreads();
		uint32_t wex = 0, tot = 0;
#pragma unroll
		for(int w2 = 0; w2 < 8; w2++) {
			const uint32_t x = sm[w2];
			if(w2 < warp)
				wex += x;
			tot += x;
		}
		if(flip)
			out[run + wex + __popc(bal & ((1u << lane) - 1u))] = e & EL_SCAF_MASK;
		run += tot;
		__syncthreads();
	}
}

__global__ void k_iota_pairs(unsigned long long* __restrict__ keys, const uint32_t* __restrict__ flip_pos, uint32_t* __restrict__ vals, const uint32_t* __restrict__ scg_scafs,
                             uint64_t K, uint32_t nd)
{
	const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
	const uint32_t d = blockIdx.y;
	if(i < K && d < nd) {
		keys[(uint64_t)d * K + i] = flip_pos[(uint64_t)d * K + i];
		vals[(uint64_t)d * K + i] = scg_scafs[i];
	}
}

}  // namespace

// ===================================================================================================
// host side
// ===================================================================================================
struct abw_search {
	abw_ctx* ctx = nullptr;
	uint64_t N = 0;
	uint32_t D = 0, S = 0, W = 1, K = 0;
	int strategy = 0;
	abw_params prm{};
	DevBuf<double> values;                    // device copy of a matrix the caller passed in host memory (a device matrix is read in place)
	DevBuf<uint64_t> rowidx;                  // matrix row of every datapoint, when the caller gave one
	ValSrc vsrc{};
	DevBuf<uint32_t> dp2scaf;
	DevBuf<uint64_t> dp_first;
	DevBuf<ScafRow> rows;
	DevBuf<uint4> frow;                       // {T, n | SCG flag << 31, length}: what k_flip_prefix gathers per flip-list entry
	DevBuf<uint64_t> scgmask;
	DevBuf<uint8_t> has_scg;
	DevBuf<uint32_t> E[2];
	DevBuf<uint32_t> scg_list[2];
	DevBuf<uint32_t> scaf_list[2];
	DevBuf<uint32_t> flip_list[2];            // sens/spec: [D][Sf] scaffolds that can flip, in the order of their flip elements, grouped by live cluster
	DevBuf<uint2> F8;                         // [D][Sf] prefix sums over the flip list of the level (k_flip_prefix)
	DevBuf<uint32_t> FC;                      // only when some scaffold has fewer datapoints in the matrix than T
	DevBuf<uint32_t> scg_k;                   // [D][K]
	bool partial = false;
	uint64_t Sf = 0;                          // scaffolds with n >= T/2+1
	DevBuf<uint8_t> assigned;
	DevBuf<double> x_gc, x_cvg;               // optional per-scaffold G+C and coverage for the terminal-bin statistics (abw_search_set_scaffold_stats)
	DevBuf<unsigned long long> xchg;          // per-level exchange buffer (side, new assignment, child statistics, ...), see search_run
	DevBuf<uint32_t> low, scaf_member, scaf_final;
	uint64_t root_totT = 0, root_totLen = 0;
	uint32_t root_viol = 0;
	std::vector<uint64_t> root_never;
	bool consumed = false;
	uint32_t max_levels = 0;                  // 0: run to the end; k: stop after k levels, the pending children become the bins
	uint32_t dim_offset = 0, dim_stride = 1, D_total = 0;     // sharded search: this object holds dimensions dim_offset + k * dim_stride (k < D) of D_total
	abw_search_profile prof{};
};

namespace {

// Device time of a family of kernels (abw_search_profile).  Only measured while the context is profiling (abw_profile_enable): stopping the
// timer waits for the device, which would keep the host from preparing the next launches of a level while the current ones run.
struct EventTimer {
	cudaEvent_t a = nullptr, b = nullptr;
	cudaStream_t st;
	bool on;
	EventTimer(cudaStream_t s, bool enabled) : st(s), on(enabled) { if(on) { cudaEventCreate(&a); cudaEventCreate(&b); } }
	~EventTimer() { if(on) { cudaEventDestroy(a); cudaEventDestroy(b); } }
	void start() { if(on) cudaEventRecord(a, st); }
	float stop() { if(!on) return 0.0f; cudaEventRecord(b, st); cudaEventSynchronize(b); float ms = 0; cudaEventElapsedTime(&ms, a, b); return ms; }
};

// ABW_TRACE=1: wall-clock milestones of abw_search_create / abw_search_run on stderr (the stream is synchronised at every milestone)
struct Trace {
	bool on;
	cudaStream_t st;
	std::chrono::steady_clock::time_point t0;
	const char* what;
	Trace(cudaStream_t s, const char* w) : on(getenv("ABW_TRACE") != nullptr), st(s), t0(std::chrono::steady_clock::now()), what(w) {}
	void mark(const char* label)
	{
		if(!on)
			return;
		cudaStreamSynchronize(st);
		const auto t1 = std::chrono::steady_clock::now();
		fprintf(stderr, "[abw trace] %s: %-28s %8.3f ms\n", what, label, std::chrono::duration<double, std::milli>(t1 - t0).count());
		t0 = t1;
	}
};

// The part of abw_search_create that starts from device arrays: s->vsrc (the matrix), d_T, d_len, s->scgmask, s->dp2scaf (when the caller gave one).
// One host wait for the whole build when all dimensions fit one chunk of sort scratch: per-scaffold tables, their validation, the root statistics, the number
// of SCG-carrying scaffolds and the key statistics of the first chunk are fetched together.
int search_build_common(abw_ctx* ctx, abw_search* s, DevBuf<uint32_t>& d_T, DevBuf<uint64_t>& d_len, bool have_dp2scaf, Trace& tr)
{
	const uint64_t N = s->N;
	const uint32_t D = s->D, S = s->S, W = s->W;
	DevBuf<uint32_t> d_scg_flag, d_scg_scafs, d_scg_index;
	DevBuf<uint64_t> d_scg_before, d_total;
	DevBuf<RootStats> d_rs;
	ABW_CUDA(ctx, d_rs.alloc(1));
	ABW_CUDA(ctx, cudaMemsetAsync(d_rs.p, 0, sizeof(RootStats), ctx->stream));
	ABW_CUDA(ctx, s->rows.alloc(S));
	ABW_CUDA(ctx, s->frow.alloc(S));
	ABW_CUDA(ctx, s->has_scg.alloc(S));
	ABW_CUDA(ctx, s->dp_first.alloc((size_t)S + 1));
	ABW_CUDA(ctx, cudaMemsetAsync(s->dp_first.p, 0, sizeof(uint64_t) * ((size_t)S + 1), ctx->stream));
	ABW_CUDA(ctx, d_scg_flag.alloc(S));
	ABW_CUDA(ctx, d_scg_before.alloc(S));
	ABW_CUDA(ctx, d_scg_index.alloc(S));
	ABW_CUDA(ctx, d_total.alloc(1));
	for(int b = 0; b < 2; b++)
		ABW_CUDA(ctx, s->scaf_list[b].alloc(S));
	if(have_dp2scaf)
		ABW_LAUNCH(ctx, k_tab_runs, abw_div_up(N, 256), 256, 0, s->dp2scaf.p, N, S, s->dp_first.p, d_rs.p);
	else {
		// no dp2scaf: the matrix holds all T datapoints of every scaffold, in scaffold order (sum(T) == N is checked with the other results below;
		// k_tab_fill_dp2scaf never writes past N)
		ABW_CHECK(abw_exclusive_scan_u32_to_u64(ctx, d_T.p, s->dp_first.p, S, s->dp_first.p + S));
		ABW_LAUNCH(ctx, k_tab_fill_dp2scaf, abw_div_up(S, 256), 256, 0, s->dp_first.p, S, N, s->dp2scaf.p);
	}
	ABW_LAUNCH(ctx, k_tab_scaffolds, abw_div_up(S, 256), 256, 0, s->dp_first.p, d_T.p, d_len.p, s->scgmask.p, S, W, s->prm.fraction_dps_in, s->rows.p, s->frow.p, s->has_scg.p,
	           d_scg_flag.p, s->scaf_list[0].p, d_rs.p);
	ABW_CHECK(abw_exclusive_scan_u32_to_u64(ctx, d_scg_flag.p, d_scg_before.p, S, d_total.p));
	// ---- per-dimension order, classes, elements; dimensions are processed in chunks to bound scratch memory
	for(int b = 0; b < 2; b++)
		ABW_CUDA(ctx, s->E[b].alloc((size_t)D * N));
	// scratch of the sort is bounded by a fixed budget (the driver is not asked for the free memory: the context caches its blocks, and the query
	// takes driver-wide locks); ABW_SORT_SCRATCH_GB overrides the 16 GB default
	const uint64_t per_dim = N * (8 + 8 + 4 + 4 + 1) + 4096;
	uint64_t budget = 16ull << 30;
	if(const char* e = getenv("ABW_SORT_SCRATCH_GB"))
		budget = std::max<uint64_t>(1, strtoull(e, nullptr, 10)) << 30;
	const uint32_t chunk = (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>(D, budget / per_dim));
	DevBuf<unsigned long long> keys, keys_tmp;
	DevBuf<uint32_t> vals, vals_tmp, flip_pos, or_and;
	DevBuf<uint8_t> cls;
	DevBuf<int> flags;                                     // [0] a value is not an exact multiple of 0.001, [1] NaN
	ABW_CUDA(ctx, flags.alloc(2));
	ABW_CUDA(ctx, or_and.alloc((size_t)2 * chunk));
	std::vector<uint32_t> h_or_and((size_t)2 * chunk);
	ABW_CUDA(ctx, keys.alloc((size_t)chunk * N));
	ABW_CUDA(ctx, keys_tmp.alloc((size_t)chunk * N));
	ABW_CUDA(ctx, vals.alloc((size_t)chunk * N));
	ABW_CUDA(ctx, vals_tmp.alloc((size_t)chunk * N));
	ABW_CUDA(ctx, cls.alloc((size_t)chunk * N));
	uint32_t* const keys32 = reinterpret_cast<uint32_t*>(keys.p);
	uint32_t* const keys32_tmp = reinterpret_cast<uint32_t*>(keys_tmp.p);
	auto launch_keys32 = [&](uint32_t d0, uint32_t nd) -> int {
		ABW_CUDA(ctx, cudaMemsetAsync(flags.p, 0, 2 * sizeof(int), ctx->stream));
		ABW_LAUNCH(ctx, k_fill_or_and, abw_div_up(nd, 256), 256, 0, or_and.p, nd);
		ABW_LAUNCH(ctx, (k_keys<true, uint32_t>), dim3(abw_div_up(N, 32), abw_div_up(nd, 32)), 256, 0, s->vsrc, N, d0, nd, keys32, vals.p, flags.p);
		// ranks inside the scaffolds on the 32-bit keys (thrown away if a value turns out not to be a multiple of 0.001), and the key bits that vary per dimension
		ABW_LAUNCH(ctx, k_rank_class<uint32_t>, dim3(abw_div_up(N, 256), nd), 256, 0, keys32, N, nd, s->dp2scaf.p, s->dp_first.p, s->rows.p, s->has_scg.p, s->strategy,
		           s->prm.fraction_dps_in, cls.p, or_and.p);
		return ABW_OK;
	};
	ABW_CHECK(launch_keys32(0, std::min(chunk, D)));
	// ---- the one host wait: tables, root statistics, SCG count, key statistics of the first chunk
	RootStats h_rs;
	uint64_t h_K = 0, sumT = N;
	int h_flags[2] = {0, 0};
	ABW_CUDA(ctx, abw_fetch(ctx, &h_rs, d_rs.p, sizeof(RootStats)));
	ABW_CUDA(ctx, abw_fetch(ctx, &h_K, d_total.p, sizeof(uint64_t)));
	if(!have_dp2scaf)
		ABW_CUDA(ctx, abw_fetch(ctx, &sumT, s->dp_first.p + S, sizeof(uint64_t)));
	ABW_CUDA(ctx, abw_fetch(ctx, h_flags, flags.p, sizeof(h_flags)));
	ABW_CUDA(ctx, abw_fetch(ctx, h_or_and.data(), or_and.p, sizeof(uint32_t) * 2 * std::min(chunk, D)));
	ABW_CUDA(ctx, abw_sync(ctx));
	if(sumT != N)
		return abw_fail(ctx, ABW_ERR_ARG, "abw_search_create: without dp2scaf the matrix must hold exactly sum(T) datapoints");
	if(h_rs.err & TB_ERR_RANGE)
		return abw_fail(ctx, ABW_ERR_ARG, "abw_search_create: dp2scaf entry out of range");
	if(h_rs.err & TB_ERR_ORDER)
		return abw_fail(ctx, ABW_ERR_ARG, "abw_search_create: datapoints must be grouped by scaffold in scaffold order (ScafDpData.cpp:91-99)");
	if(h_rs.err & TB_ERR_T)
		return abw_fail(ctx, ABW_ERR_ARG, "abw_search_create: every scaffold needs T >= 2 datapoints (ScafDpData.cpp:92-93 drops the others)");
	if(h_rs.err & TB_ERR_COUNT)
		return abw_fail(ctx, ABW_ERR_ARG, "abw_search_create: every scaffold needs between 1 and T datapoints in the matrix");
	s->root_totT = h_rs.totT;
	s->root_totLen = h_rs.totLen;
	s->root_viol = h_rs.viol;
	s->Sf = h_rs.Sf;
	s->partial = h_rs.partial != 0;
	s->root_never.assign(h_rs.never, h_rs.never + W);
	if(s->root_totT >= (1ull << 31))
		return abw_fail(ctx, ABW_ERR_UNSUPPORTED, "abw_search_create: sum of T over scaffolds must be below 2^31");
	s->K = (uint32_t)h_K;
	const uint64_t K = s->K;
	tr.mark("tables and first keys");
	ABW_CUDA(ctx, d_scg_scafs.alloc(std::max<uint64_t>(K, 1)));
	ABW_LAUNCH(ctx, k_tab_scg, abw_div_up(S, 256), 256, 0, d_scg_flag.p, d_scg_before.p, S, d_scg_index.p, d_scg_scafs.p);
	for(int b = 0; b < 2; b++)
		ABW_CUDA(ctx, s->scg_list[b].alloc((size_t)D * K));
	ABW_CUDA(ctx, flip_pos.alloc((size_t)D * K));
	for(uint32_t d0 = 0; d0 < D; d0 += chunk) {
		const uint32_t nd = std::min(chunk, D - d0);
		const dim3 grid(abw_div_up(N, 256), nd);
		if(d0 > 0) {
			ABW_CHECK(launch_keys32(d0, nd));
			ABW_CUDA(ctx, abw_fetch(ctx, h_flags, flags.p, sizeof(h_flags)));
			ABW_CUDA(ctx, abw_fetch(ctx, h_or_and.data(), or_and.p, sizeof(uint32_t) * 2 * nd));
			ABW_CUDA(ctx, abw_sync(ctx));
		}
		uint32_t* fp = (s->strategy == ABW_SENS_SPEC && K > 0)? flip_pos.p + (uint64_t)d0 * K : nullptr;
		if(!h_flags[0]) {
			// one digit plan per run of dimensions that need the same number of passes (k-mer thousandths fit one digit, coverage needs two)
			auto passes = [](uint32_t varying) { int best = 64; for(int wd = 8; wd <= 9; wd++) { int c = 0, bit = 0; while(bit < 32) { if(!((varying >> bit) & 1u)) { bit++; continue; } c++; bit += wd; } best = std::min(best, c); } return best; };
			for(uint32_t r0 = 0; r0 < nd;) {
				uint32_t vary = h_or_and[2 * r0] ^ h_or_and[2 * r0 + 1];
				const int p0 = passes(vary);
				uint32_t r1 = r0 + 1;
				while(r1 < nd) {
					const uint32_t vd = h_or_and[2 * r1] ^ h_or_and[2 * r1 + 1];
					if(passes(vd) != p0 || passes(vary | vd) != p0)
						break;
					vary |= vd;
					r1++;
				}
				ABW_CHECK(abw_radix_sort_pairs_u32_varying(ctx, keys32 + (uint64_t)r0 * N, keys32_tmp + (uint64_t)r0 * N, vals.p + (uint64_t)r0 * N, vals_tmp.p + (uint64_t)r0 * N, N,
				                                           r1 - r0, N, (unsigned long long)vary));
				r0 = r1;
			}
			ABW_LAUNCH(ctx, k_pack_elements<uint32_t>, grid, 256, 0, keys32, vals.p, N, nd, s->dp2scaf.p, cls.p, s->E[0].p + (uint64_t)d0 * N, d_scg_index.p, fp, K);
		}
		else {
			// arbitrary doubles: 64-bit order-preserving keys
			ABW_LAUNCH(ctx, (k_keys<false, unsigned long long>), dim3(abw_div_up(N, 32), abw_div_up(nd, 32)), 256, 0, s->vsrc, N, d0, nd, keys.p, vals.p, flags.p);
			ABW_LAUNCH(ctx, k_rank_class<unsigned long long>, grid, 256, 0, keys.p, N, nd, s->dp2scaf.p, s->dp_first.p, s->rows.p, s->has_scg.p, s->strategy,
			           s->prm.fraction_dps_in, cls.p, (uint32_t*)nullptr);
			ABW_CHECK(abw_radix_sort_pairs_u64(ctx, (uint64_t*)keys.p, (uint64_t*)keys_tmp.p, vals.p, vals_tmp.p, N, nd, N, 64));
			ABW_LAUNCH(ctx, k_pack_elements<unsigned long long>, grid, 256, 0, keys.p, vals.p, N, nd, s->dp2scaf.p, cls.p, s->E[0].p + (uint64_t)d0 * N, d_scg_index.p, fp, K);
			int h_nan[2] = {0, 0};
			ABW_CUDA(ctx, abw_fetch(ctx, h_nan, flags.p, sizeof(h_nan)));
			ABW_CUDA(ctx, abw_sync(ctx));
			if(h_nan[1])
				return abw_fail(ctx, ABW_ERR_ARG, "abw_search_create: NaN in the feature matrix (comp_by_value is not a strict weak order on NaN)");
		}
	}
	tr.mark("classes, sort, elements");
	keys.release(); keys_tmp.release(); vals.release(); vals_tmp.release(); cls.release();
	// ---- per-dimension flip list: every scaffold that can flip has exactly one class-1 element per dimension
	if(s->strategy == ABW_SENS_SPEC && s->Sf > 0) {
		const uint64_t Sf = s->Sf;
		for(int b = 0; b < 2; b++)
			ABW_CUDA(ctx, s->flip_list[b].alloc((size_t)D * Sf));
		ABW_CUDA(ctx, s->F8.alloc((size_t)D * Sf));
		if(s->partial)
			ABW_CUDA(ctx, s->FC.alloc((size_t)D * Sf));
		ABW_CUDA(ctx, s->scg_k.alloc((size_t)D * std::max<uint64_t>(K, 1)));
		const uint32_t tiles = abw_div_up(N, SW_TILE);
		DevBuf<uint32_t> counts;
		ABW_CUDA(ctx, counts.alloc((size_t)D * tiles));
		ABW_LAUNCH(ctx, k_flip_count, dim3(tiles, D), 256, 0, s->E[0].p, N, tiles, counts.p);
		ABW_LAUNCH(ctx, k_flip_write, dim3(tiles, D), 256, 0, s->E[0].p, N, tiles, counts.p, s->flip_list[0].p, Sf);
	}
	tr.mark("flip lists");
	// ---- per-dimension list of SCG-carrying scaffolds in the order their flip element appears
	if(s->strategy == ABW_SENS_SPEC && K > 0) {
		DevBuf<unsigned long long> lk, lk_tmp;
		DevBuf<uint32_t> lv_tmp;
		ABW_CUDA(ctx, lk.alloc((size_t)D * K));
		ABW_CUDA(ctx, lk_tmp.alloc((size_t)D * K));
		ABW_CUDA(ctx, lv_tmp.alloc((size_t)D * K));
		dim3 grid(abw_div_up(K, 256), D);
		ABW_LAUNCH(ctx, k_iota_pairs, grid, 256, 0, lk.p, flip_pos.p, s->scg_list[0].p, d_scg_scafs.p, K, D);
		int nbits = 1;
		while(nbits < 32 && (1ull << nbits) < N)
			nbits++;
		// positions spread over [0, N): every bit below nbits is taken as varying, which saves the inspection pass and its host round trip
		ABW_CHECK(abw_radix_sort_pairs_u64(ctx, (uint64_t*)lk.p, (uint64_t*)lk_tmp.p, s->scg_list[0].p, lv_tmp.p, K, D, K, -nbits));
	}
	tr.mark("SCG lists");
	// ---- root cluster (its scaffold list 0..S-1 was written by k_tab_scaffolds)
	ABW_CUDA(ctx, s->assigned.alloc(S));
	ABW_CUDA(ctx, s->low.alloc(S));
	ABW_CUDA(ctx, s->scaf_member.alloc(S));
	ABW_CUDA(ctx, s->scaf_final.alloc(S));
	ABW_CUDA(ctx, cudaMemsetAsync(s->assigned.p, 1, S, ctx->stream));
	ABW_CUDA(ctx, cudaMemsetAsync(s->low.p, 0, sizeof(uint32_t) * S, ctx->stream));
	ABW_CUDA(ctx, cudaMemsetAsync(s->scaf_member.p, 0, sizeof(uint32_t) * S, ctx->stream));
	ABW_CUDA(ctx, cudaMemsetAsync(s->scaf_final.p, 0, sizeof(uint32_t) * S, ctx->stream));
	tr.mark("root cluster");
	return ABW_OK;                                         // later entry points work in the order of the context stream: no wait here
}

// abw_search_create: the caller's host arrays go to the device, the matrix is read where it lies (a host matrix is uploaded once, in its own layout)
int search_build(abw_ctx* ctx, abw_search* s, const double* values, int values_on_device, int layout, uint64_t ld, uint64_t nrows, const uint64_t* h_row_of_dp,
                 const uint32_t* h_dp2scaf, const uint32_t* h_T, const uint64_t* h_len, const uint64_t* h_scgmask)
{
	const uint64_t N = s->N;
	const uint32_t D = s->D, S = s->S, W = s->W;
	Trace tr(ctx->stream, "create");
	ABW_CUDA(ctx, s->dp2scaf.alloc(N));
	if(h_dp2scaf)
		ABW_CUDA(ctx, cudaMemcpyAsync(s->dp2scaf.p, h_dp2scaf, sizeof(uint32_t) * N, cudaMemcpyHostToDevice, ctx->stream));
	ABW_CUDA(ctx, s->scgmask.alloc((size_t)S * W));
	if(h_scgmask)
		ABW_CUDA(ctx, cudaMemcpyAsync(s->scgmask.p, h_scgmask, sizeof(uint64_t) * (size_t)S * W, cudaMemcpyHostToDevice, ctx->stream));
	else
		ABW_CUDA(ctx, cudaMemsetAsync(s->scgmask.p, 0, sizeof(uint64_t) * (size_t)S * W, ctx->stream));
	DevBuf<uint32_t> d_T;
	DevBuf<uint64_t> d_len;
	ABW_CUDA(ctx, d_T.alloc(S));
	ABW_CUDA(ctx, d_len.alloc(S));
	ABW_CUDA(ctx, cudaMemcpyAsync(d_T.p, h_T, sizeof(uint32_t) * S, cudaMemcpyHostToDevice, ctx->stream));
	ABW_CUDA(ctx, cudaMemcpyAsync(d_len.p, h_len, sizeof(uint64_t) * S, cudaMemcpyHostToDevice, ctx->stream));
	s->vsrc.p = values; s->vsrc.ld = ld; s->vsrc.layout = layout; s->vsrc.rowidx = nullptr;
	if(h_row_of_dp) {
		for(uint64_t i = 0; i < N; i++)
			if(h_row_of_dp[i] >= nrows)
				return abw_fail(ctx, ABW_ERR_ARG, "abw_search_create: row_of_dp entry out of range");
		ABW_CUDA(ctx, s->rowidx.alloc(N));
		ABW_CUDA(ctx, cudaMemcpyAsync(s->rowidx.p, h_row_of_dp, sizeof(uint64_t) * N, cudaMemcpyHostToDevice, ctx->stream));
		s->vsrc.rowidx = s->rowidx.p;
	}
	if(!values_on_device) {
		const uint64_t count = (layout == ABW_LAYOUT_ROWMAJOR)? nrows * ld : (uint64_t)D * ld;
		ABW_CUDA(ctx, s->values.alloc(count));
		ABW_CUDA(ctx, cudaMemcpyAsync(s->values.p, values, sizeof(double) * count, cudaMemcpyHostToDevice, ctx->stream));
		s->vsrc.p = s->values.p;
	}
	tr.mark("uploads");
	ABW_CHECK(search_build_common(ctx, s, d_T, d_len, h_dp2scaf != nullptr, tr));
	// the caller's host arrays (pageable memory: the driver staged them) may be reused as soon as the call returns; the uploads are complete then
	// because the build waited for the stream after they were enqueued
	return ABW_OK;
}

// one thread per scaffold of the assembly: windows per scaffold, and whether ScafDpData keeps it (at least two windows, ScafDpData.cpp:92-93)
__global__ void k_feat_counts(const uint64_t* __restrict__ seg_first, uint32_t nscaf, uint32_t* __restrict__ keep, uint32_t* __restrict__ cnt)
{
	const uint32_t sidx = blockIdx.x * blockDim.x + threadIdx.x;
	if(sidx >= nscaf)
		return;
	const uint64_t c = seg_first[sidx + 1] - seg_first[sidx];
	const bool k = c >= 2;
	keep[sidx] = k? 1u : 0u;
	cnt[sidx] = k? (uint32_t)c : 0u;
}
__global__ void k_feat_gather(const uint64_t* __restrict__ seg_first, uint32_t nscaf, const uint32_t* __restrict__ keep, const uint64_t* __restrict__ newidx,
                              const uint64_t* __restrict__ dpfirst, const uint32_t* __restrict__ cnt, const uint64_t* __restrict__ len_in, const uint64_t* __restrict__ mask_in,
                              uint32_t W, uint32_t* __restrict__ T_out, uint64_t* __restrict__ len_out, uint64_t* __restrict__ mask_out, uint64_t* __restrict__ rowidx,
                              uint32_t* __restrict__ kept_out)
{
	const uint32_t sidx = blockIdx.x * blockDim.x + threadIdx.x;
	if(sidx >= nscaf || !keep[sidx])
		return;
	const uint64_t ns = newidx[sidx];
	T_out[ns] = cnt[sidx];
	len_out[ns] = len_in[sidx];
	for(uint32_t w = 0; w < W; w++)
		mask_out[ns * W + w] = mask_in? mask_in[(uint64_t)sidx * W + w] : 0ull;
	kept_out[ns] = sidx;
	const uint64_t f = dpfirst[sidx], r0 = seg_first[sidx];
	for(uint32_t j = 0; j < cnt[sidx]; j++)
		rowidx[f + j] = r0 + j;
}

// Replaces the work-list loop abawaca.cpp:98-197.  The host enqueues level after level on the context stream and never waits for one: work sizes live in the
// device-resident LevelCtl, every kernel is launched with a grid that does not depend on the data (its CTAs walk the level's work items), look-back words carry
// the level's epoch instead of being cleared per level, and k_level_decide reports progress through mapped pinned memory, which the host polls between launches.
// A sharded search (coll != null) adds two collectives per level -- the per-cluster bests of all ranks, then one buffer with the owner's vote -- whose sizes are
// bounds known to the host (at level l at most 2^l clusters), so they are enqueued blindly as well when the collectives are stream ordered.
int search_run(abw_ctx* ctx, abw_search* s, const abw_collectives* coll, abw_cluster_rec* h_recs, uint32_t cap, uint32_t* nrecs, uint32_t* h_dp2cluster,
               uint32_t* h_scaf2cluster)
{
	const uint32_t world = coll? (uint32_t)coll->world : 1u;
	const bool ordered = coll && coll->stream_ordered != 0;
	if(s->D_total == 0)
		s->D_total = s->D;
	const uint64_t N = s->N;
	const uint32_t D = s->D, S = s->S, W = s->W, K = s->K;
	const uint64_t Sf = s->Sf;
	const abw_params& prm = s->prm;
	const bool ss = s->strategy == ABW_SENS_SPEC;
	if(s->consumed)
		return abw_fail(ctx, ABW_ERR_ARG, "abw_search_run: this search object was already run (element arrays are consumed); create a new one");
	s->consumed = true;
	EventTimer tm(ctx->stream, ctx->profiling);
	s->prof.sweep_ms = s->prof.partition_ms = s->prof.other_ms = 0;
	s->prof.sweep_elements = s->prof.partition_elements = 0;
	s->prof.levels = s->prof.sweep_launches = 0;

	SweepParams sp;
	sp.thr = prm.cluster_ndps_threshold;
	// candidates below min_reported_score are not examined; that must never hide a candidate is_legal would accept, so the cut is never above
	// the caller's product threshold (a caller who lowers product_threshold and leaves min_reported_score alone still gets every legal split)
	sp.min_score = ss? std::min(prm.min_reported_score, prm.product_threshold) : prm.min_reported_score;
	sp.prune = (float)(sp.min_score * (1.0 - 1e-5));
	if(!(sp.prune > 0.0f))
		sp.prune = 0.0f;
	sp.scg_min_size = prm.scg_min_size;
	sp.fraction_in = prm.fraction_dps_in;

	// ---- bounds: clusters of one level (every cluster below the root holds at least cluster_ndps_threshold datapoints), tiles, splits
	const uint64_t thr = std::max<uint32_t>(prm.cluster_ndps_threshold, 1);
	const uint64_t Cmax64 = 2 * (N / thr) + 2;
	if(Cmax64 >= (1ull << 31))
		return abw_fail(ctx, ABW_ERR_UNSUPPORTED, "abw_search_run: too many clusters per level for this build");
	const uint32_t Cmax = (uint32_t)Cmax64, Pmax = Cmax / 2 + 1;
	const uint64_t TTmax = N / SW_TILE + Cmax + 1, FPTmax = Sf / FP_TILE + Cmax + 1;
	const uint64_t items_max = TTmax * D, fp_items_max = ss? FPTmax * D : 0;
	const uint64_t part_tab_max = (S + N + Sf + K) / SW_TILE + 4ull * Pmax + 8;
	const uint64_t part_items_max = (S / SW_TILE + Pmax + 1) + (N / SW_TILE + Pmax + 1) * D + (ss? (Sf / SW_TILE + Pmax + 1) * D + (K / SW_TILE + Pmax + 1) * D : 0);
	if(items_max >= (1ull << 31) || part_items_max >= (1ull << 31))
		return abw_fail(ctx, ABW_ERR_UNSUPPORTED, "abw_search_run: more than 2^31 tiles in one level");
	const uint64_t lb_words = std::max(items_max, part_items_max);
	const uint64_t tab_total_max = (uint64_t)K + Cmax;

	// ---- buffers of the run
	DevBuf<LevelCtl> d_ctl;
	DevBuf<LevelCluster> d_cl[2];
	DevBuf<CandRec> d_cand, d_best, d_best_all;
	DevBuf<SplitJob> d_jobs;
	DevBuf<uint32_t> d_jobs_mine, d_job_of, d_status;
	DevBuf<abw_best> d_bestrec;
	DevBuf<uint2> d_cl_tab, d_ss_tab, d_tile_tab, d_fp_tab, d_part_tab, d_tm_tab, d_klohi;
	DevBuf<PartJob> d_part_jobs;
	DevBuf<TermJob> d_tjobs;
	DevBuf<TermStats> d_tstats;
	DevBuf<uint64_t> d_tunion, d_suffix;
	DevBuf<abw_cluster_rec> d_recs;
	DevBuf<AggSlot> d_aggs, d_prefixes;
	DevBuf<unsigned long long> d_lookback;
	DevBuf<uint8_t> d_tab;
	ABW_CUDA(ctx, d_ctl.alloc(1));
	for(int b = 0; b < 2; b++)
		ABW_CUDA(ctx, d_cl[b].alloc(Cmax));
	ABW_CUDA(ctx, d_cand.alloc(items_max));
	ABW_CUDA(ctx, d_best.alloc(Cmax));
	if(world > 1)
		ABW_CUDA(ctx, d_best_all.alloc((size_t)Cmax * world));
	ABW_CUDA(ctx, d_jobs.alloc(Cmax));
	ABW_CUDA(ctx, d_jobs_mine.alloc(Cmax));
	ABW_CUDA(ctx, d_job_of.alloc(Cmax));
	ABW_CUDA(ctx, d_bestrec.alloc(Cmax));
	ABW_CUDA(ctx, d_cl_tab.alloc(N / CL_CHUNK + Cmax + 1));
	ABW_CUDA(ctx, d_ss_tab.alloc(S / SS_CHUNK + Cmax + 1));
	ABW_CUDA(ctx, d_tile_tab.alloc(TTmax));
	ABW_CUDA(ctx, d_fp_tab.alloc(ss? FPTmax : 1));
	ABW_CUDA(ctx, d_part_tab.alloc(part_tab_max));
	ABW_CUDA(ctx, d_tm_tab.alloc(S / TM_CHUNK + Cmax + 1));
	ABW_CUDA(ctx, d_part_jobs.alloc((size_t)4 * Pmax));
	ABW_CUDA(ctx, d_tjobs.alloc(Cmax));
	ABW_CUDA(ctx, d_tstats.alloc(Cmax));
	ABW_CUDA(ctx, d_tunion.alloc((size_t)Cmax * W));
	const uint32_t rec_cap = h_recs? cap : 0;
	ABW_CUDA(ctx, d_recs.alloc(std::max<uint32_t>(rec_cap, 1)));
	ABW_CUDA(ctx, d_lookback.alloc(lb_words));
	ABW_CUDA(ctx, cudaMemsetAsync(d_lookback.p, 0, sizeof(unsigned long long) * lb_words, ctx->stream));
	const uint64_t st_items = ss? fp_items_max : items_max;            // status / aggregate slots: flip-prefix tiles (sens/spec) or sweep tiles (split-scafs)
	ABW_CUDA(ctx, d_status.alloc(std::max<uint64_t>(st_items, 1)));
	ABW_CUDA(ctx, d_aggs.alloc(std::max<uint64_t>(st_items, 1)));
	ABW_CUDA(ctx, d_prefixes.alloc(std::max<uint64_t>(st_items, 1)));
	ABW_CUDA(ctx, cudaMemsetAsync(d_status.p, 0, sizeof(uint32_t) * std::max<uint64_t>(st_items, 1), ctx->stream));
	if(ss) {
		ABW_CUDA(ctx, d_tab.alloc((size_t)D * tab_total_max));
		ABW_CUDA(ctx, d_klohi.alloc((size_t)D * Cmax));
		ABW_CUDA(ctx, d_suffix.alloc((size_t)D * std::max<uint32_t>(K, 1) * W));
	}
	// what the owner of a winning dimension produces for everybody, in one buffer so that a sharded search needs one sum per level:
	//   side bytes | assignment bytes | child statistics [J][2] | separating-value keys [J] | masks of scaffolds that can never flip [J][2][W]
	const size_t s8 = ((size_t)S + 7) / 8, stat_words = sizeof(ChildStats) / 8;
	auto xwords_for = [&](uint64_t Jb) { return 2 * s8 + (size_t)Jb * (2 * stat_words + 1 + 2 * W); };
	if(s->xchg.n < xwords_for(Cmax))
		ABW_CUDA(ctx, s->xchg.alloc(xwords_for(Cmax)));
	ABW_CUDA(ctx, cudaMemsetAsync(s->xchg.p, 0, sizeof(unsigned long long) * xwords_for(Cmax), ctx->stream));
	uint8_t* const d_side = reinterpret_cast<uint8_t*>(s->xchg.p);
	uint8_t* const d_new_assigned = d_side + 8 * s8;

	// progress words in mapped pinned memory (one block per context)
	if(!ctx->h_prog) {
		ABW_CUDA(ctx, cudaHostAlloc((void**)&ctx->h_prog, 256, cudaHostAllocMapped));
	}
	LevelProgress* const h_prog = reinterpret_cast<LevelProgress*>(ctx->h_prog);
	h_prog->levels_done = 0; h_prog->done = 0; h_prog->error = 0; h_prog->ticks = 0; h_prog->done_at = 0;

	// ---- root cluster and control block
	{
		LevelCluster root;
		memset(&root, 0, sizeof(root));
		root.id = 1;
		root.parent = 0;
		root.d.off = 0;
		root.d.n = (uint32_t)N;
		root.d.kOff = 0; root.d.K = K; root.d.tabOff = 0;
		root.d.sOff = 0; root.d.ns = S;
		root.d.totT = (uint32_t)s->root_totT;
		root.d.U = S;
		root.d.totLen = s->root_totLen;
		root.d.ss_ok = (s->root_viol == 0);
		root.d.tile0 = 0;
		root.d.fOff = 0; root.d.nf = (uint32_t)Sf;
		root.nassigned = S;
		for(uint32_t w = 0; w < W && w < s->root_never.size(); w++)
			root.never[w] = s->root_never[w];
		LevelCtl c0;
		memset(&c0, 0, sizeof(c0));
		c0.C = 1;
		c0.TT = abw_div_up(N, SW_TILE);
		c0.FPT = (ss && Sf > 0)? abw_div_up(Sf, FP_TILE) : 0;
		c0.tab_total = K + 1;
		c0.next_id = 2;
		std::vector<uint2> tt(c0.TT), ft(std::max<uint32_t>(c0.FPT, 1));
		for(uint32_t t = 0; t < c0.TT; t++) tt[t] = make_uint2(0, t);
		for(uint32_t t = 0; t < c0.FPT; t++) ft[t] = make_uint2(0, t);
		ABW_CUDA(ctx, abw_upload_small(ctx, d_cl[0].p, &root, sizeof(root)));
		ABW_CUDA(ctx, abw_upload_small(ctx, d_ctl.p, &c0, sizeof(c0)));
		ABW_CUDA(ctx, abw_upload_small(ctx, d_tile_tab.p, tt.data(), sizeof(uint2) * c0.TT));
		if(c0.FPT)
			ABW_CUDA(ctx, abw_upload_small(ctx, d_fp_tab.p, ft.data(), sizeof(uint2) * c0.FPT));
	}
	LevelBufs B;
	memset(&B, 0, sizeof(B));
	B.ctl = d_ctl.p;
	ABW_CUDA(ctx, cudaHostGetDevicePointer((void**)&B.prog, ctx->h_prog, 0));
	B.cl[0] = d_cl[0].p; B.cl[1] = d_cl[1].p;
	B.best = d_best.p; B.best_all = d_best_all.p;
	B.jobs = d_jobs.p; B.jobs_mine = d_jobs_mine.p; B.job_of = d_job_of.p; B.bestrec = d_bestrec.p;
	B.cl_tab = d_cl_tab.p; B.ss_tab = d_ss_tab.p; B.tile_tab = d_tile_tab.p; B.fp_tab = d_fp_tab.p; B.part_tab = d_part_tab.p; B.tm_tab = d_tm_tab.p;
	B.part_jobs = d_part_jobs.p; B.tjobs = d_tjobs.p; B.tstats = d_tstats.p; B.tunion = d_tunion.p;
	B.recs = d_recs.p; B.rec_cap = rec_cap; B.Cmax = Cmax; B.Pmax = Pmax;
	B.low = s->low.p;

	// grids: CTAs walk the work items of a level, whatever their number turns out to be
	const unsigned int sms = (unsigned int)ctx->sm_count;
	const unsigned int g_sweep = (unsigned int)std::min<uint64_t>(items_max, (uint64_t)sms * SWEEP_CTAS), g_fp = (unsigned int)std::min<uint64_t>(std::max<uint64_t>(fp_items_max, 1), (uint64_t)sms * FLIP_CTAS);
	const unsigned int g_part = (unsigned int)std::min<uint64_t>(part_items_max, (uint64_t)sms * PART_CTAS), g_small = sms * 4;

	// levels the host may run ahead of the device.  A sharded search must make the same number of collective calls on every rank, so there the decision
	// to enqueue level l is a function of device state that is final when it is read: level l is enqueued iff the search had not ended by level
	// l - lead (every rank waits until that level has been reported, then reads done_at, which is written once).  That enqueues lead - 1 empty levels
	// (kernels that find no work, collectives over zeroes) after the last one, on every rank alike, and hides the host's round trip behind the
	// kernels of lead - 1 levels.
	const uint32_t lead = (world > 1)? 3u : 6u;
	// side stream for k_finalize_terminal (not while kernels are timed one by one); its destructor makes the main stream wait, so that no buffer of this
	// call returns to the block cache while a side kernel may still use it
	struct SideStream {
		abw_ctx* ctx;
		bool on = false, pending = false;
		cudaError_t join()
		{
			if(!pending)
				return cudaSuccess;
			pending = false;
			return cudaStreamWaitEvent(ctx->stream, ctx->ev_join, 0);
		}
		~SideStream() { join(); }
	} side{ctx};
	if(!ctx->profiling) {
		if(!ctx->side_stream) {
			ABW_CUDA(ctx, cudaStreamCreateWithFlags(&ctx->side_stream, cudaStreamNonBlocking));
			ABW_CUDA(ctx, cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming));
			ABW_CUDA(ctx, cudaEventCreateWithFlags(&ctx->ev_join, cudaEventDisableTiming));
		}
		side.on = true;
	}
	uint32_t lvl = 0;
	uint64_t Cb_seen = ~0ull;
	bool finished = false;
	int cur = 0;
	const uint32_t max_levels = s->max_levels;
	while(!finished) {
		if(max_levels > 0 && lvl >= max_levels)
			break;
		const bool last_level = max_levels > 0 && lvl + 1 >= max_levels;
		const uint32_t ep_sweep = 2 * lvl + 1, ep_part = 2 * lvl + 2;
		if(lvl > 0 && lvl % 16 == 0) {
			// the packed look-back words hold 6 bits of the epoch: clear them before an epoch can repeat
			ABW_CUDA(ctx, cudaMemsetAsync(d_lookback.p, 0, sizeof(unsigned long long) * lb_words, ctx->stream));
		}
		// at level l there are at most 2^l clusters, and at most 2^(lead-1) times those of the last level whose verdict every rank has waited for:
		// the host-known bound for the collectives of a sharded search (the same on every rank)
		const uint32_t Cb = (uint32_t)std::min<uint64_t>(std::min<uint64_t>(Cmax, Cb_seen), (lvl < 31)? (1ull << lvl) : Cmax);
		ChildStats* const d_stats = reinterpret_cast<ChildStats*>(s->xchg.p + 2 * s8);
		unsigned long long* const d_value_key = s->xchg.p + 2 * s8 + (size_t)Cb * 2 * stat_words;
		uint64_t* const d_child_never = reinterpret_cast<uint64_t*>(d_value_key + Cb);
		const size_t xwords = xwords_for(Cb);
		if(world > 1)          // bytes of earlier levels would otherwise be summed again; without ranks to sum over, every byte that is read was written in this level
			ABW_CUDA(ctx, cudaMemsetAsync(s->xchg.p, 0, sizeof(unsigned long long) * 2 * s8, ctx->stream));
		tm.start();
		if(ss) {
			ABW_LAUNCH(ctx, k_pass_table, g_small, PT_WARPS * 32, 0, s->scg_list[cur].p, (uint64_t)K, d_cl[cur].p, d_ctl.p, s->scgmask.p, W, prm.scg_overlap_threshold,
			           d_suffix.p, d_tab.p, D, d_klohi.p, Cmax, (unsigned long long)prm.scg_min_size);
			s->prof.other_ms += tm.stop();
			tm.start();
			if(Sf > 0)
				ABW_LAUNCH(ctx, k_flip_prefix, g_fp, SW_THREADS, 0, s->flip_list[cur].p, Sf, d_cl[cur].p, D, d_ctl.p, d_fp_tab.p, s->frow.p, ep_sweep, d_status.p,
				           d_aggs.p, d_prefixes.p, s->F8.p, s->FC.p, s->scg_k.p, (uint64_t)K, d_klohi.p, Cmax, (unsigned long long)prm.scg_min_size);
			ABW_LAUNCH(ctx, k_sweep_ss, g_sweep, SW_THREADS, 0, s->E[cur].p, N, d_cl[cur].p, D, d_ctl.p, d_tile_tab.p, s->F8.p, s->FC.p, s->scg_k.p, (uint64_t)K, d_klohi.p, Cmax,
			           Sf, d_tab.p, sp, ep_sweep, d_lookback.p, d_cand.p);
		}
		else
			ABW_LAUNCH(ctx, k_sweep_split_scafs, g_sweep, SW_THREADS, 0, s->E[cur].p, N, d_cl[cur].p, D, d_ctl.p, d_tile_tab.p, s->rows.p, sp,
			           ep_sweep, d_status.p, d_aggs.p, d_prefixes.p, d_cand.p);
		s->prof.sweep_ms += tm.stop();
		tm.start();
		if(ss)
			ABW_LAUNCH(ctx, k_reduce_best<ABW_SENS_SPEC>, g_small, RB_THREADS, 0, d_cand.p, D, d_ctl.p, d_cl[cur].p, s->dim_offset, s->dim_stride, d_best.p);
		else
			ABW_LAUNCH(ctx, k_reduce_best<ABW_SPLIT_SCAFS>, g_small, RB_THREADS, 0, d_cand.p, D, d_ctl.p, d_cl[cur].p, s->dim_offset, s->dim_stride, d_best.p);
		if(world > 1) {
			// the per-rank best of every cluster, gathered; k_level_jobs applies the same total order on every rank
			if(!ordered)
				ABW_CUDA(ctx, abw_sync(ctx));
			if(coll->allgather(coll->user, d_best.p, d_best_all.p, sizeof(CandRec) * Cb) != 0)
				return abw_fail(ctx, ABW_ERR_CUDA, "abw_search_run_sharded: allgather callback failed");
		}
		ABW_LAUNCH(ctx, k_level_jobs, 1, LV_THREADS, 0, B, cur, world, Cb, s->strategy, prm, s->dim_offset, s->dim_stride, D, s->E[cur].p, N, d_stats, d_value_key, d_child_never, W);
		ABW_LAUNCH(ctx, k_count_low, g_small, 256, 0, s->E[cur].p, N, B, cur, s->dim_offset, s->dim_stride, s->low.p);
		ABW_LAUNCH(ctx, k_scaf_sides, g_small * 2, SS_CHUNK, 0, s->scaf_list[cur].p, B, cur, s->dim_offset, s->dim_stride, s->rows.p, s->low.p, s->dp_first.p, s->vsrc, s->scgmask.p, W,
		           s->strategy, prm.fraction_dps_in, d_side, d_new_assigned, d_stats, d_child_never, d_value_key);
		if(world > 1) {
			// every quantity is non-zero on exactly one rank (the owner of the winning dimension): a sum is a gather
			if(!ordered)
				ABW_CUDA(ctx, abw_sync(ctx));
			if(coll->allreduce_sum_i64(coll->user, s->xchg.p, xwords) != 0)
				return abw_fail(ctx, ABW_ERR_CUDA, "abw_search_run_sharded: allreduce callback failed");
		}
		const uint32_t pd0 = 1, pd1 = last_level? 0u : D, pd2 = (!last_level && ss && Sf > 0)? D : 0u, pd3 = (!last_level && ss && K > 0)? D : 0u;
		ABW_CUDA(ctx, side.join());                            // k_finalize_terminal of the previous level (side stream) has to be through with the job tables
		ABW_LAUNCH(ctx, k_level_decide, 1, LV_THREADS, 0, B, cur, s->strategy, prm, D, W, s->dim_offset, pd0, pd1, pd2, pd3, last_level? 0 : 1, d_stats, d_value_key,
		           d_child_never);
		if(side.on) {
			// the terminal clusters of this level are finished beside the partition: nothing on the main stream reads what k_finalize_terminal writes
			// (bins, tallies, fields of the terminal records) or overwrites what it reads (job tables of the level, scaffold list [cur], the `assigned`
			// bytes of terminal clusters' scaffolds -- the partition commits those of SPLIT clusters) before k_level_decide of the NEXT level, which waits
			ABW_CUDA(ctx, cudaEventRecord(ctx->ev_fork, ctx->stream));
			ABW_CUDA(ctx, cudaStreamWaitEvent(ctx->side_stream, ctx->ev_fork, 0));
			k_finalize_terminal<<<g_small, 128, 0, ctx->side_stream>>>(s->scaf_list[cur].p, B, s->rows.p, s->assigned.p, s->scgmask.p, W, s->scaf_member.p, s->scaf_final.p,
			                                                            (const double*)s->x_gc.p, (const double*)s->x_cvg.p);
			ctx->launches++;
			ABW_CUDA(ctx, cudaGetLastError());
			ABW_CUDA(ctx, cudaEventRecord(ctx->ev_join, ctx->side_stream));
			side.pending = true;
		}
		else
			ABW_LAUNCH(ctx, k_finalize_terminal, g_small, 128, 0, s->scaf_list[cur].p, B, s->rows.p, s->assigned.p, s->scgmask.p, W, s->scaf_member.p, s->scaf_final.p,
			           (const double*)s->x_gc.p, (const double*)s->x_cvg.p);
		s->prof.other_ms += tm.stop();
		tm.start();
		{
			PartPlans pp;
			pp.in[0] = s->scaf_list[cur].p; pp.out[0] = s->scaf_list[cur ^ 1].p; pp.stride[0] = S;
			pp.in[1] = s->E[cur].p; pp.out[1] = s->E[cur ^ 1].p; pp.stride[1] = N;
			pp.in[2] = s->flip_list[cur].p; pp.out[2] = s->flip_list[cur ^ 1].p; pp.stride[2] = Sf;
			pp.in[3] = s->scg_list[cur].p; pp.out[3] = s->scg_list[cur ^ 1].p; pp.stride[3] = K;
			ABW_LAUNCH(ctx, k_partition2, g_part, SW_THREADS, 0, pp, d_ctl.p, d_part_jobs.p, d_part_tab.p, d_side, d_new_assigned, s->assigned.p, ep_part, d_lookback.p);
		}
		s->prof.partition_ms += tm.stop();
		cur ^= 1;
		lvl++;
		// progress: stop as soon as the device has reported the last level; never run more than `lead` levels ahead of it
		while(true) {
			if(world > 1) {
				// deterministic on every rank: levels 0 .. lvl - lead must have been reported before level lvl is enqueued
				if(lvl < lead)
					break;
				const uint32_t need = lvl - lead + 1, tk = h_prog->ticks;
				__sync_synchronize();
				if(tk >= need) {
					const uint32_t da = h_prog->done_at;
					finished = h_prog->error != 0 || (da != 0 && da <= need);
					// clusters of level `need` (written once, by the level before it), doubled for every level enqueued since
					Cb_seen = (uint64_t)h_prog->c_next[(need - 1) & 15u] << (lvl - need);
					break;
				}
			}
			else {
				const uint32_t ld = h_prog->levels_done;        // written after `done`: a level that is reported has its verdict visible
				__sync_synchronize();
				if(h_prog->error) {
					finished = true;
					break;
				}
				if(ld >= lvl) {                                 // the level just enqueued has been decided
					finished = h_prog->done != 0;
					break;
				}
				if(h_prog->done) {                              // an earlier level was the last one: what was enqueued since is empty
					finished = true;
					break;
				}
				if(lvl - ld < lead)
					break;
			}
			if(cudaStreamQuery(ctx->stream) == cudaSuccess) {
				// the stream is idle although a level has not been reported: a kernel fault surfaces here
				ABW_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
				__sync_synchronize();
				if(h_prog->ticks < lvl && !h_prog->done)
					return abw_fail(ctx, ABW_ERR_CUDA, "abw_search_run: internal error, the device stopped reporting levels");
			}
		}
	}
	ABW_CUDA(ctx, side.join());
	ABW_CUDA(ctx, abw_sync(ctx));
	LevelCtl h_ctl;
	ABW_CUDA(ctx, abw_fetch(ctx, &h_ctl, d_ctl.p, sizeof(h_ctl)));
	ABW_CUDA(ctx, abw_sync(ctx));
	if(h_ctl.error == 2)
		return abw_fail(ctx, ABW_ERR_CUDA, "abw_search_run: internal error, more clusters in a level than the bound");
	if(h_ctl.error)
		return abw_fail(ctx, ABW_ERR_CUDA, "abw_search_run: internal error, a look-back wait timed out");
	if(!h_ctl.done && max_levels > 0 && h_ctl.level >= max_levels && h_ctl.P > 0) {
		// level limit reached: the pending clusters (the children written by the last level) are reported as bins (their ids) without being evaluated
		ABW_LAUNCH(ctx, k_pending_jobs, 1, LV_THREADS, 0, B, cur, W);
		ABW_LAUNCH(ctx, k_finalize_terminal, g_small, 128, 0, s->scaf_list[cur].p, B, s->rows.p, s->assigned.p, s->scgmask.p, W, s->scaf_member.p, s->scaf_final.p,
		           (const double*)nullptr, (const double*)nullptr);
	}
	s->prof.levels = h_ctl.level;
	s->prof.sweep_launches = h_ctl.sweep_launches;
	s->prof.sweep_elements = h_ctl.sweep_elements;
	s->prof.partition_elements = h_ctl.partition_elements;
	const uint32_t nrec = h_ctl.nrec;
	if(nrecs)
		*nrecs = nrec;
	if(h_recs && std::min(nrec, cap) > 0)
		ABW_CUDA(ctx, abw_fetch(ctx, h_recs, d_recs.p, sizeof(abw_cluster_rec) * std::min(nrec, cap)));
	if(h_scaf2cluster)
		ABW_CUDA(ctx, abw_fetch(ctx, h_scaf2cluster, s->scaf_final.p, sizeof(uint32_t) * S));
	if(h_dp2cluster) {
		DevBuf<uint32_t> d_dp;
		ABW_CUDA(ctx, d_dp.alloc(N));
		ABW_LAUNCH(ctx, k_dp_bins, abw_div_up(N, 256), 256, 0, s->dp2scaf.p, s->scaf_member.p, N, d_dp.p);
		ABW_CUDA(ctx, abw_fetch(ctx, h_dp2cluster, d_dp.p, sizeof(uint32_t) * N));
		ABW_CUDA(ctx, abw_sync(ctx));
	}
	ABW_CUDA(ctx, abw_sync(ctx));
	return ABW_OK;
}

}  // namespace

extern "C" {

int abw_search_create(abw_ctx* ctx, const double* values, int values_on_device, int layout, uint64_t ld, uint64_t nrows, const uint64_t* h_row_of_dp,
                      uint64_t N, uint32_t D, const uint32_t* h_dp2scaf, uint32_t S, const uint32_t* h_T, const uint64_t* h_len, const uint64_t* h_scgmask, uint32_t W,
                      const abw_params* params, int strategy, abw_search** out)
{
	if(!ctx || !out || !values || !h_T || !h_len || (W > 0 && !h_scgmask))
		return abw_fail(ctx, ABW_ERR_ARG, "abw_search_create: null argument");
	if(strategy != ABW_SENS_SPEC && strategy != ABW_SPLIT_SCAFS)
		return abw_fail(ctx, ABW_ERR_ARG, "abw_search_create: unknown strategy");
	if(N == 0 || D == 0 || S == 0)
		return abw_fail(ctx, ABW_ERR_ARG, "abw_search_create: empty problem");
	if(W > SCG_WMAX)
		return abw_fail(ctx, ABW_ERR_UNSUPPORTED, "abw_search_create: at most 512 distinct SCG names (W <= 8)");
	if(N >= (1ull << 28) || S >= (1u << EL_SCAF_BITS))       // the look-back words of the sweep carry two 28-bit counts (cnt_payload)
		return abw_fail(ctx, ABW_ERR_UNSUPPORTED, "abw_search_create: at most 2^28-1 datapoints and 2^27-1 scaffolds per device");
	if(!h_row_of_dp)
		nrows = N;
	if(layout != ABW_LAYOUT_COLMAJOR && layout != ABW_LAYOUT_ROWMAJOR && layout != ABW_LAYOUT_ROWMAJOR_MILLI32)
		return abw_fail(ctx, ABW_ERR_ARG, "abw_search_create: unknown layout");
	if(layout == ABW_LAYOUT_ROWMAJOR_MILLI32 && !values_on_device)
		return abw_fail(ctx, ABW_ERR_UNSUPPORTED, "abw_search_create: a matrix of integer thousandths must be in device memory");
	if(nrows < 1 || (layout == ABW_LAYOUT_COLMAJOR && ld < nrows) || (layout != ABW_LAYOUT_COLMAJOR && ld < D))
		return abw_fail(ctx, ABW_ERR_ARG, "abw_search_create: leading dimension too small");
	ABW_ENTER(ctx);
	abw_search* s = new abw_search();
	s->ctx = ctx;
	s->N = N; s->D = D; s->S = S; s->W = (W == 0)? 1 : W;
	s->strategy = strategy;
	if(params)
		s->prm = *params;
	else
		abw_default_params(&s->prm);
	EventTimer tm(ctx->stream, ctx->profiling);
	tm.start();
	int rc = search_build(ctx, s, values, values_on_device, layout, ld, nrows, h_row_of_dp, h_dp2scaf, h_T, h_len, (W > 0)? h_scgmask : nullptr);
	s->prof.build_ms = tm.stop();
	if(rc != ABW_OK) {
		delete s;
		return rc;
	}
	*out = s;
	return ABW_OK;
}

// The search problem of a feature build without a trip through the host: T = windows per scaffold, scaffolds with fewer than two windows dropped
// (ScafDpData.cpp:92-93), datapoints = the rows of the kept scaffolds in row order.
int abw_search_create_from_features(abw_ctx* ctx, const abw_segments* g, const double* d_rows, uint64_t ld, uint32_t D, const uint64_t* h_len, const uint64_t* h_scgmask,
                                    uint32_t W, const abw_params* params, int strategy, uint32_t* S_out, uint64_t* N_out, uint32_t* h_kept, abw_search** out)
{
	if(!ctx || !g || !d_rows || !h_len || !out || (W > 0 && !h_scgmask))
		return abw_fail(ctx, ABW_ERR_ARG, "abw_search_create_from_features: null argument");
	if(strategy != ABW_SENS_SPEC && strategy != ABW_SPLIT_SCAFS)
		return abw_fail(ctx, ABW_ERR_ARG, "abw_search_create_from_features: unknown strategy");
	if(W > SCG_WMAX)
		return abw_fail(ctx, ABW_ERR_UNSUPPORTED, "abw_search_create: at most 512 distinct SCG names (W <= 8)");
	if(D == 0 || ld < D || g->nscaf == 0 || g->nseg == 0)
		return abw_fail(ctx, ABW_ERR_ARG, "abw_search_create_from_features: empty problem or row stride too small");
	ABW_ENTER(ctx);
	const uint32_t nscaf = g->nscaf, Wd = (W == 0)? 1 : W;
	abw_search* s = new abw_search();
	s->ctx = ctx;
	s->D = D; s->W = Wd;
	s->strategy = strategy;
	if(params)
		s->prm = *params;
	else
		abw_default_params(&s->prm);
	EventTimer tm(ctx->stream, ctx->profiling);
	tm.start();
	int rc = [&]() -> int {
		Trace tr(ctx->stream, "create");
		DevBuf<uint32_t> keep, cnt, d_T, d_kept;
		DevBuf<uint64_t> newidx, dpfirst, totals, len_in, mask_in, d_len;
		ABW_CUDA(ctx, keep.alloc(nscaf));
		ABW_CUDA(ctx, cnt.alloc(nscaf));
		ABW_CUDA(ctx, newidx.alloc(nscaf));
		ABW_CUDA(ctx, dpfirst.alloc(nscaf));
		ABW_CUDA(ctx, totals.alloc(2));
		ABW_CUDA(ctx, len_in.alloc(nscaf));
		ABW_CUDA(ctx, cudaMemcpyAsync(len_in.p, h_len, sizeof(uint64_t) * nscaf, cudaMemcpyHostToDevice, ctx->stream));
		if(W > 0) {
			ABW_CUDA(ctx, mask_in.alloc((size_t)nscaf * W));
			ABW_CUDA(ctx, cudaMemcpyAsync(mask_in.p, h_scgmask, sizeof(uint64_t) * (size_t)nscaf * W, cudaMemcpyHostToDevice, ctx->stream));
		}
		ABW_LAUNCH(ctx, k_feat_counts, abw_div_up(nscaf, 256), 256, 0, g->seg_first.p, nscaf, keep.p, cnt.p);
		ABW_CHECK(abw_exclusive_scan_u32_to_u64(ctx, keep.p, newidx.p, nscaf, totals.p));
		ABW_CHECK(abw_exclusive_scan_u32_to_u64(ctx, cnt.p, dpfirst.p, nscaf, totals.p + 1));
		uint64_t h_tot[2] = {0, 0};
		ABW_CUDA(ctx, abw_fetch(ctx, h_tot, totals.p, sizeof(h_tot)));
		ABW_CUDA(ctx, abw_sync(ctx));
		const uint64_t S = h_tot[0], N = h_tot[1];
		if(S == 0 || N == 0)
			return abw_fail(ctx, ABW_ERR_ARG, "abw_search_create_from_features: no scaffold has two windows");
		if(N >= (1ull << 28) || S >= (1u << EL_SCAF_BITS))
			return abw_fail(ctx, ABW_ERR_UNSUPPORTED, "abw_search_create: at most 2^28-1 datapoints and 2^27-1 scaffolds per device");
		s->N = N; s->S = (uint32_t)S;
		ABW_CUDA(ctx, d_T.alloc(S));
		ABW_CUDA(ctx, d_len.alloc(S));
		ABW_CUDA(ctx, d_kept.alloc(S));
		ABW_CUDA(ctx, s->scgmask.alloc((size_t)S * Wd));
		ABW_CUDA(ctx, s->rowidx.alloc(N));
		ABW_CUDA(ctx, s->dp2scaf.alloc(N));
		ABW_LAUNCH(ctx, k_feat_gather, abw_div_up(nscaf, 256), 256, 0, g->seg_first.p, nscaf, keep.p, newidx.p, dpfirst.p, cnt.p, len_in.p, (const uint64_t*)mask_in.p, Wd,
		           d_T.p, d_len.p, s->scgmask.p, s->rowidx.p, d_kept.p);
		if(h_kept)
			ABW_CUDA(ctx, abw_fetch(ctx, h_kept, d_kept.p, sizeof(uint32_t) * S));     // handed over at the wait inside the build
		s->vsrc.p = d_rows; s->vsrc.ld = ld; s->vsrc.layout = ABW_LAYOUT_ROWMAJOR;
		s->vsrc.rowidx = (S == nscaf)? nullptr : s->rowidx.p;                          // nothing dropped: datapoint i is row i
		tr.mark("problem from the feature build");
		ABW_CHECK(search_build_common(ctx, s, d_T, d_len, false, tr));
		if(S_out) *S_out = (uint32_t)S;
		if(N_out) *N_out = N;
		return ABW_OK;
	}();
	s->prof.build_ms = tm.stop();
	if(rc != ABW_OK) {
		delete s;
		return rc;
	}
	*out = s;
	return ABW_OK;
}

void abw_search_destroy(abw_search* s) { delete s; }

int abw_search_run(abw_ctx* ctx, abw_search* s, abw_cluster_rec* h_recs, uint32_t cap, uint32_t* nrecs, uint32_t* h_dp2cluster, uint32_t* h_scaf2cluster)
{
	if(!ctx || !s)
		return abw_fail(ctx, ABW_ERR_ARG, "abw_search_run: null argument");
	ABW_ENTER(ctx);
	return search_run(ctx, s, nullptr, h_recs, cap, nrecs, h_dp2cluster, h_scaf2cluster);
}

int abw_search_set_scaffold_stats(abw_ctx* ctx, abw_search* s, const double* h_gc, const double* h_cvg)
{
	if(!ctx || !s || !h_gc || !h_cvg)
		return abw_fail(ctx, ABW_ERR_ARG, "abw_search_set_scaffold_stats: null argument");
	ABW_ENTER(ctx);
	ABW_CUDA(ctx, s->x_gc.alloc(s->S));
	ABW_CUDA(ctx, s->x_cvg.alloc(s->S));
	ABW_CUDA(ctx, cudaMemcpyAsync(s->x_gc.p, h_gc, sizeof(double) * s->S, cudaMemcpyHostToDevice, ctx->stream));
	ABW_CUDA(ctx, cudaMemcpyAsync(s->x_cvg.p, h_cvg, sizeof(double) * s->S, cudaMemcpyHostToDevice, ctx->stream));
	ABW_CUDA(ctx, abw_sync(ctx));
	return ABW_OK;
}

int abw_search_set_max_levels(abw_search* s, uint32_t max_levels)
{
	if(!s)
		return ABW_ERR_ARG;
	s->max_levels = max_levels;
	return ABW_OK;
}

int abw_search_set_shard(abw_search* s, uint32_t dim_offset, uint32_t D_total)
{
	return abw_search_set_shard_strided(s, dim_offset, 1, D_total);
}

int abw_search_set_shard_strided(abw_search* s, uint32_t dim_offset, uint32_t dim_stride, uint32_t D_total)
{
	if(!s || dim_stride == 0 || (s->D > 0 && (uint64_t)dim_offset + (uint64_t)(s->D - 1) * dim_stride >= D_total))
		return ABW_ERR_ARG;
	s->dim_offset = dim_offset;
	s->dim_stride = dim_stride;
	s->D_total = D_total;
	return ABW_OK;
}

int abw_search_run_sharded(abw_ctx* ctx, abw_search* s, const abw_collectives* coll, abw_cluster_rec* h_recs, uint32_t cap, uint32_t* nrecs, uint32_t* h_dp2cluster,
                           uint32_t* h_scaf2cluster)
{
	if(!ctx || !s || !coll || !coll->allgather || !coll->allreduce_sum_i64 || coll->world < 1 || coll->rank < 0 || coll->rank >= coll->world)
		return abw_fail(ctx, ABW_ERR_ARG, "abw_search_run_sharded: bad argument");
	ABW_ENTER(ctx);
	return search_run(ctx, s, coll, h_recs, cap, nrecs, h_dp2cluster, h_scaf2cluster);
}

int abw_search_get_profile(const abw_search* s, abw_search_profile* out)
{
	if(!s || !out)
		return ABW_ERR_ARG;
	*out = s->prof;
	return ABW_OK;
}

int abw_cluster_scg(abw_ctx* ctx, const abw_search* s, const uint32_t* h_scafs, uint32_t nscafs, uint32_t* nunique, double* avg)
{
	if(!ctx || !s || (!h_scafs && nscafs))
		return abw_fail(ctx, ABW_ERR_ARG, "abw_cluster_scg: null argument");
	ABW_ENTER(ctx);
	// SCGdb::num_unique_scgs / average_num_copies_for_unique_scgs (SCGdb.cpp:6-18,41-55)
	DevBuf<uint32_t> d_list;
	DevBuf<TermStats> d_st;
	DevBuf<uint64_t> d_un;
	for(uint32_t i = 0; i < nscafs; i++)
		if(h_scafs[i] >= s->S)
			return abw_fail(ctx, ABW_ERR_ARG, "abw_cluster_scg: scaffold index out of range");
	// the reference walks a std::set of scaffolds: a scaffold listed twice counts once
	std::vector<uint32_t> set(h_scafs, h_scafs + nscafs);
	std::sort(set.begin(), set.end());
	set.erase(std::unique(set.begin(), set.end()), set.end());
	nscafs = (uint32_t)set.size();
	ABW_CUDA(ctx, d_list.alloc(nscafs));
	ABW_CUDA(ctx, d_st.alloc(1));
	ABW_CUDA(ctx, d_un.alloc(s->W));
	if(nscafs)
		ABW_CUDA(ctx, cudaMemcpyAsync(d_list.p, set.data(), sizeof(uint32_t) * nscafs, cudaMemcpyHostToDevice, ctx->stream));
	ABW_CUDA(ctx, cudaMemsetAsync(d_st.p, 0, sizeof(TermStats), ctx->stream));
	ABW_CUDA(ctx, cudaMemsetAsync(d_un.p, 0, sizeof(uint64_t) * s->W, ctx->stream));
	if(nscafs)
		ABW_LAUNCH(ctx, k_scg_tally, std::min<unsigned int>(abw_div_up(nscafs, 128), 1024u), 128, 0, d_list.p, nscafs, s->scgmask.p, s->W, d_st.p, d_un.p);
	TermStats ts;
	std::vector<uint64_t> un(s->W);
	ABW_CUDA(ctx, abw_fetch(ctx, &ts, d_st.p, sizeof(ts)));
	ABW_CUDA(ctx, abw_fetch(ctx, un.data(), d_un.p, sizeof(uint64_t) * s->W));
	ABW_CUDA(ctx, abw_sync(ctx));
	uint32_t u = 0;
	for(uint32_t w = 0; w < s->W; w++)
		u += (uint32_t)__builtin_popcountll(un[w]);
	if(nunique) *nunique = u;
	if(avg) *avg = (ts.scg_copies == 0)? 0 : (double)ts.scg_copies / (double)u;
	return ABW_OK;
}

}  // extern "C"
