// Per-sample coverage of abawaca-build on the device: Scaf::add_mapped_read / Scaf_segment::add_mapped_read (abawaca-build.cpp:177-185, 231-244)
// behind the read filter of the SAM loop (:546-551).
//
// The reference adds fl(overlap_i / window length) in SAM order (an order-dependent fp64 sum, quirk Q5) and prints int(1000 * sum) / 1000.0.
// Formulation here (DESIGN.md section 4):
//   pass 1  k_cov_sum       one pass over the read records: window(s) of every read by arithmetic on a 16-byte scaffold record, overlap added to a
//                           64-bit integer sum per (sample, window).  The overlaps of a tile of 1024 reads are first combined in a shared-memory
//                           table indexed by window (shared atomics): one global atomic per touched window and tile instead of one per read.  Every
//                           tile also leaves the range of windows it touched.
//           k_cov_quotient  one thread per (sample, window): where the truncation to three decimals cannot depend on the order of the reads the value
//                           follows from the integer sum alone; the other windows (the exact value IS a multiple of 0.001, or a huge sum) are flagged.
//   pass 2  k_cov_pairs     only tiles whose window range holds a flagged window are read again; their (flagged window, overlap) pairs of ALL samples are
//                           sorted stably by (sample, window) in one radix sort and summed in SAM order by one thread per window.
// ABW_FEAT_RAW (un-truncated doubles) sends every pair through pass 2.
// Two record formats: abw_read (16 bytes, filter applied here) and abw_read8 (8 bytes: reads the host parser already filtered, SURVEY.md section 8b(4)).
// Samples of coordinate-sorted reads (ABW_READS_SORTED, about 2 bytes per read) are decoded into abw_read8 records first (readcodec.cu).
#include "features.cuh"
#include <algorithm>

namespace {

constexpr uint32_t FULL = 0xffffffffu;
constexpr int COV_ITEMS = 4;                                // consecutive reads per thread
constexpr int COV_THREADS = 256;
constexpr int COV_TILE = COV_THREADS * COV_ITEMS;

struct ReadSrc {
	const void*           p;        // abw_read[n] or abw_read8[n]
	unsigned long long    n;
	const unsigned short* len16;    // compact format: per-read lengths, or null: every read is `len` long
	uint32_t              len;
	int32_t               fmt;      // ABW_READS_FULL | ABW_READS_COMPACT
	uint32_t              tile0;    // index of the sample's first tile in the per-tile arrays of the batch
	uint32_t              ntiles;
};

struct Rd4 {
	uint32_t scaf[COV_ITEMS], pos0[COV_ITEMS], len[COV_ITEMS];
	bool     acc[COV_ITEMS];
};

// COV_ITEMS consecutive reads of a thread; acc = the read counts (abawaca-build.cpp:546-550: mapped, at most max_snps mismatches, not a secondary
// alignment, scaffold known).  Compact records were filtered by the host; their scaffold index is still checked.
__device__ __forceinline__ void load_reads4(const ReadSrc& src, uint64_t r0, uint32_t max_snps, uint32_t nscaf, Rd4& rd)
{
	if(src.fmt == ABW_READS_FULL) {
		const uint4* __restrict__ p = reinterpret_cast<const uint4*>(src.p);
#pragma unroll
		for(int j = 0; j < COV_ITEMS; j++) {
			uint4 x = make_uint4(0xFFFFFFFFu, 0, 0, 0);
			if(r0 + j < src.n)
				x = __ldg(p + r0 + j);                          // scaf, pos0, len, flag | nsnps << 16
			const uint32_t flag = x.w & 0xFFFFu, nsnps = x.w >> 16;
			rd.scaf[j] = x.x; rd.pos0[j] = x.y; rd.len[j] = x.z;
			rd.acc[j] = !((flag & 0x4u) || (nsnps > max_snps) || (flag & 0x100u)) && x.x < nscaf;
		}
	}
	else {
		const uint2* __restrict__ p = reinterpret_cast<const uint2*>(src.p);
		uint2 x[COV_ITEMS];
		if(r0 + COV_ITEMS <= src.n && (reinterpret_cast<uintptr_t>(p) & 15u) == 0) {
			const uint4 a = __ldg(reinterpret_cast<const uint4*>(p + r0)), b = __ldg(reinterpret_cast<const uint4*>(p + r0 + 2));
			x[0] = make_uint2(a.x, a.y); x[1] = make_uint2(a.z, a.w); x[2] = make_uint2(b.x, b.y); x[3] = make_uint2(b.z, b.w);
		}
		else {
#pragma unroll
			for(int j = 0; j < COV_ITEMS; j++)
				x[j] = (r0 + j < src.n)? __ldg(p + r0 + j) : make_uint2(0xFFFFFFFFu, 0);
		}
#pragma unroll
		for(int j = 0; j < COV_ITEMS; j++) {
			rd.scaf[j] = x[j].x; rd.pos0[j] = x[j].y;
			rd.len[j] = (src.len16 != nullptr && r0 + j < src.n)? (uint32_t)__ldg(src.len16 + r0 + j) : src.len;
			rd.acc[j] = x[j].x < nscaf;
		}
	}
}

// The windows a read overlaps, in order: window w of a scaffold counts when s0 <= end(w) && e0 >= start(w) with the 0-based read positions
// s0 = POS - 1, e0 = s0 + len - 1 against the 1-based window bounds (quirk Q3, abawaca-build.cpp:182-183, 233-237; kept as it is).
// A scaffold without N (COV_REGULAR) has the windows [l nbps + 1, (l + 1) nbps]: arithmetic only.  Otherwise the window is guessed as
// (s0 - 1) / nbps, verified against the window ends and, next to runs of N, found by binary search; windows of a scaffold are contiguous
// (start = previous end + 1, first start = 1), so only the ends are read.
struct WinIter {
	uint32_t g, f1;                 // current window; one past the last window of the scaffold
	uint64_t st, en;                // bounds of the current window
	uint64_t s, e;                  // the read
	uint32_t nb;                    // bases per window of a regular scaffold, 0: look the ends up
	const uint64_t* __restrict__ ends;

	__device__ __forceinline__ void init(uint32_t pos0, uint32_t len, const uint4 si, const uint64_t* __restrict__ seg_end)
	{
		s = pos0;
		e = (uint64_t)pos0 + len - 1;
		ends = seg_end;
		const uint32_t f0 = si.x;
		f1 = si.x + si.y;
		if(si.w == COV_REGULAR) {
			nb = si.z;
			const uint32_t q = pos0? (pos0 - 1) / nb : 0u;     // position s >= 1 lies in window (s - 1) / nbps; position 0 before the first one
			if(q >= si.y) {                                     // behind the last window (the trailing bases no window holds)
				g = f1; st = 1; en = 0;
				return;
			}
			g = f0 + q;
			st = (uint64_t)q * nb + 1;
			en = st + nb - 1;
			return;
		}
		nb = 0;
		uint32_t q = 0;
		if(pos0 > 0 && si.w == 0)
			q = (pos0 - 1) / max(si.z, 1u);                     // an all-N scaffold (nbps 0) has one window per character
		uint32_t gg = f0 + min(si.y - 1u, q);
		uint64_t cur_end = __ldg(seg_end + gg), prev_end = (gg > f0)? __ldg(seg_end + gg - 1) : 0ull;
		if(!((gg == f0 || prev_end < s) && cur_end >= s)) {
			uint32_t lo = f0, hi = f1;                          // runs of N moved the boundaries: first window whose end is >= s
			while(lo < hi) {
				const uint32_t mid = lo + ((hi - lo) >> 1);
				if(__ldg(seg_end + mid) < s) lo = mid + 1; else hi = mid;
			}
			gg = lo;
			cur_end = (gg < f1)? __ldg(seg_end + gg) : 0ull;
			prev_end = (gg > f0)? __ldg(seg_end + gg - 1) : 0ull;
		}
		g = gg;
		st = prev_end + 1;                                      // first window of a scaffold: prev_end is 0 and the start 1
		en = cur_end;
	}
	__device__ __forceinline__ bool valid() const { return g < f1 && !(e < st); }
	__device__ __forceinline__ uint32_t overlap() const
	{
		const uint64_t s2 = (s < st)? st : s, e2 = (e > en)? en : e;
		return (uint32_t)(e2 - s2 + 1);
	}
	__device__ __forceinline__ void next()
	{
		g++;
		st = en + 1;
		if(nb)
			en = st + nb - 1;
		else if(g < f1)
			en = __ldg(ends + g);
	}
};

// The common case of WinIter in 32-bit arithmetic and without a loop: a read of 1 <= len < 2^20 bases at pos0 < 2^31 - 2^20 on a scaffold without N
// (windows [q nb + 1, (q + 1) nb]) that reaches at most two windows.  Returns false when the general walk is needed; else ov1 (0: the read counts for
// no window) belongs to window g and ov2 (0: none) to window g + 1.
__device__ __forceinline__ bool regular_two(const uint4 si, uint32_t pos0, uint32_t len, uint32_t& g, uint32_t& ov1, uint32_t& ov2)
{
	g = 0; ov1 = 0; ov2 = 0;
	if(!(si.w == COV_REGULAR && pos0 < 0x7FF00000u && len - 1u < (1u << 20) - 1u))
		return false;
	const uint32_t nb = si.z, cnt = si.y;
	const uint32_t q = pos0? (pos0 - 1u) / nb : 0u;
	const uint32_t st = q * nb + 1u, en = st + nb - 1u, e = pos0 + len - 1u;
	if(!(q < cnt && e >= st))
		return true;
	if(e > en + nb && q + 2u < cnt)
		return false;                                           // a third window: rare, left to the general walk
	g = si.x + q;
	ov1 = min(e, en) - max(pos0, st) + 1u;
	if(e > en && q + 1u < cnt)
		ov2 = min(e - en, nb);
	return true;
}

// dst[key] += v for the lanes with `valid`, one atomic per distinct key of the warp.  Every lane of the warp calls it.  (Used where it runs once per
// thread; in the hot loop of k_cov_sum the per-group reduction of a non-uniform mask compiles to a loop over the groups and was the bottleneck.)
__device__ __forceinline__ void warp_add_by_key(unsigned long long* __restrict__ dst, uint32_t key, uint32_t v, bool valid)
{
	if(__any_sync(FULL, valid && v >= (1u << 26))) {           // a 32-bit warp sum could overflow: plain atomics (reads are never that long in practice)
		if(valid)
			atomicAdd(&dst[key], (unsigned long long)v);
		return;
	}
	const uint32_t peers = __match_any_sync(FULL, valid? key : 0xFFFFFFFFu);
	const uint32_t sum = __reduce_add_sync(peers, valid? v : 0u);
	if(valid && (threadIdx.x & 31) == (uint32_t)(__ffs(peers) - 1))
		atomicAdd(&dst[key], (unsigned long long)sum);
}

// pass 1: integer sum of the overlaps per window (order free), window range of every tile, per-scaffold read bases of the -c sample (:242-243).
// A tile of 1024 consecutive reads of a SAM file in scaffold or coordinate order touches a handful of neighbouring windows: the overlaps are first
// added up in a shared-memory table indexed by (window - lowest window of the tile) with shared atomics, and every touched window then costs ONE
// 64-bit global atomic per tile.  Windows beyond the table (reads in no particular order) and overlaps of 2^20 bases or more go to global memory directly.
constexpr uint32_t CS_RANGE = 2048;                         // windows per tile held in shared memory
constexpr uint32_t CS_SCAFS = 512;                          // scaffolds per tile held in shared memory (-c sample only)
constexpr uint32_t CS_MAX_OV = 1u << 20;                    // 2048 overlaps below 2^20 cannot overflow a 32-bit table entry

template <bool NBPS>
__global__ void __launch_bounds__(COV_THREADS, 4) k_cov_sum(const ReadSrc src, uint32_t max_snps, uint32_t nscaf, const uint4* __restrict__ scaf_info,
                                                           const uint64_t* __restrict__ seg_end, unsigned long long* __restrict__ sum_ov,
                                                           uint2* __restrict__ tile_range, unsigned long long* __restrict__ scaf_nbps)
{
	abw_grid_wait();
	__shared__ uint32_t sm_acc[CS_RANGE];
	__shared__ uint32_t sm_nb[NBPS? CS_SCAFS : 1];
	__shared__ uint32_t sm_min, sm_max, sm_smin;
	for(uint32_t i = threadIdx.x; i < CS_RANGE; i += COV_THREADS)
		sm_acc[i] = 0;
	if(NBPS)
		for(uint32_t i = threadIdx.x; i < CS_SCAFS; i += COV_THREADS)
			sm_nb[i] = 0;
	if(threadIdx.x == 0) {
		sm_min = 0xFFFFFFFFu;
		sm_max = 0;
		sm_smin = 0xFFFFFFFFu;
	}
	__syncthreads();
	const uint64_t r0 = ((uint64_t)blockIdx.x * COV_THREADS + threadIdx.x) * COV_ITEMS;
	Rd4 rd;
	load_reads4(src, r0, max_snps, nscaf, rd);
	uint4 si[COV_ITEMS];
#pragma unroll
	for(int j = 0; j < COV_ITEMS; j++)
		si[j] = rd.acc[j]? __ldg(scaf_info + rd.scaf[j]) : make_uint4(0, 0, 1, 0);
	// first and second window of every read; further windows (reads longer than a window: rare) go to global memory at once
	uint32_t g1[COV_ITEMS], ov1[COV_ITEMS], ov2[COV_ITEMS];    // ov == 0: no such window (an overlap is at least 1)
	uint32_t gmin = 0xFFFFFFFFu, gmax = 0, smin = 0xFFFFFFFFu;
#pragma unroll
	for(int j = 0; j < COV_ITEMS; j++) {
		g1[j] = 0; ov1[j] = 0; ov2[j] = 0;
		if(NBPS && rd.acc[j])
			smin = min(smin, rd.scaf[j]);
		if(!(rd.acc[j] && si[j].y > 0))
			continue;
		const uint32_t pos0 = rd.pos0[j], len = rd.len[j];
		if(si[j].w == COV_REGULAR && pos0 < 0x7FF00000u && len - 1u < CS_MAX_OV - 1u) {
			// the common case in 32-bit arithmetic and without a loop: a scaffold without N has the windows [q nb + 1, (q + 1) nb] (WinIter::init /
			// next / overlap for COV_REGULAR, specialised; 1 <= len < 2^20 and pos0 < 2^31 - 2^20 keep every quantity below 2^32)
			const uint32_t nb = si[j].z, cnt = si[j].y;
			const uint32_t q = pos0? (pos0 - 1u) / nb : 0u;
			const uint32_t st = q * nb + 1u, en = st + nb - 1u, e = pos0 + len - 1u;
			if(q < cnt && e >= st) {
				const uint32_t g = si[j].x + q;
				g1[j] = g;
				ov1[j] = min(e, en) - max(pos0, st) + 1u;
				gmin = min(gmin, g);
				gmax = max(gmax, g);
				if(e > en && q + 1u < cnt) {
					ov2[j] = min(e - en, nb);
					gmax = max(gmax, g + 1u);
					// a read longer than a window reaches further windows (rare)
					uint32_t gg = g + 2u, stt = en + nb + 1u;
					while(gg < si[j].x + cnt && e >= stt) {
						atomicAdd(&sum_ov[gg], (unsigned long long)min(e - stt + 1u, nb));
						gmax = max(gmax, gg);
						gg++;
						stt += nb;
					}
				}
			}
			continue;
		}
		WinIter it;
		it.init(pos0, len, si[j], seg_end);
		if(!it.valid())
			continue;
		g1[j] = it.g;
		ov1[j] = it.overlap();
		gmin = min(gmin, it.g);
		gmax = max(gmax, it.g);
		it.next();
		if(it.valid()) {
			ov2[j] = it.overlap();
			gmax = max(gmax, it.g);
			for(it.next(); it.valid(); it.next()) {
				atomicAdd(&sum_ov[it.g], (unsigned long long)it.overlap());
				gmax = max(gmax, it.g);
			}
		}
	}
	gmin = __reduce_min_sync(FULL, gmin);
	gmax = __reduce_max_sync(FULL, gmax);
	if(NBPS)
		smin = __reduce_min_sync(FULL, smin);
	if((threadIdx.x & 31) == 0) {
		if(gmin <= gmax) {
			atomicMin(&sm_min, gmin);
			atomicMax(&sm_max, gmax);
		}
		if(NBPS && smin != 0xFFFFFFFFu)
			atomicMin(&sm_smin, smin);
	}
	__syncthreads();
	const uint32_t base = sm_min, top = sm_max, sbase = sm_smin;
	if(threadIdx.x == 0)
		tile_range[src.tile0 + blockIdx.x] = make_uint2(base, top);        // base > top: the tile touches no window
#pragma unroll
	for(int j = 0; j < COV_ITEMS; j++) {
		if(NBPS && rd.acc[j]) {
			const uint32_t rel = rd.scaf[j] - sbase;
			if(rel < CS_SCAFS && rd.len[j] < CS_MAX_OV)
				atomicAdd(&sm_nb[rel], rd.len[j]);
			else
				atomicAdd(&scaf_nbps[rd.scaf[j]], (unsigned long long)rd.len[j]);
		}
		if(ov1[j]) {
			const uint32_t rel = g1[j] - base;
			if(rel < CS_RANGE && ov1[j] < CS_MAX_OV)
				atomicAdd(&sm_acc[rel], ov1[j]);
			else
				atomicAdd(&sum_ov[g1[j]], (unsigned long long)ov1[j]);
		}
		if(ov2[j]) {
			const uint32_t rel = g1[j] + 1 - base;
			if(rel < CS_RANGE && ov2[j] < CS_MAX_OV)
				atomicAdd(&sm_acc[rel], ov2[j]);
			else
				atomicAdd(&sum_ov[g1[j] + 1], (unsigned long long)ov2[j]);
		}
	}
	__syncthreads();
	if(base <= top) {
		const uint32_t n = min(top - base + 1, CS_RANGE);
		for(uint32_t i = threadIdx.x; i < n; i += COV_THREADS) {
			const uint32_t v = sm_acc[i];
			if(v)
				atomicAdd(&sum_ov[base + i], (unsigned long long)v);
		}
	}
	if(NBPS && sbase != 0xFFFFFFFFu)
		for(uint32_t i = threadIdx.x; i < CS_SCAFS && sbase + i < nscaf; i += COV_THREADS) {
			const uint32_t v = sm_nb[i];
			if(v)
				atomicAdd(&scaf_nbps[sbase + i], (unsigned long long)v);
		}
}

// one thread per (sample, window): the value from the integer sum where the truncation cannot depend on the order of the reads, a flag elsewhere.
// With A = sum of the overlaps, the exact value of 1000 * sum is 1000 A / len = m + r / len (0 <= r < len).  The floating-point sum of n <= A terms is
// within (n + 1) u A / len of A / len (u = 2^-53: one rounding per quotient, per addition and for the product with 1000), so the product the reference
// truncates lies within E = 1000 (A + 1) u A / len of m + r / len; whenever r != 0 and E < min(r, len - r) / len the truncation is m whatever the order
// was (the test is made with twice that bound).  Windows with r == 0 (the rounding direction decides) or a sum beyond 2^40 are flagged.
__global__ void __launch_bounds__(256) k_cov_quotient(const unsigned long long* __restrict__ sum_ov, uint64_t nseg, const uint64_t* __restrict__ seg_start,
                                                      const uint64_t* __restrict__ seg_end, double* __restrict__ rows, uint64_t ld, uint32_t col0,
                                                      uint32_t* __restrict__ flag_bits, uint32_t nwords, uint32_t* __restrict__ nflagged)
{
	abw_grid_wait();
	const uint64_t g = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
	const uint32_t sample = blockIdx.y;
	bool f = false;
	if(g < nseg) {
		const uint64_t A = sum_ov[(uint64_t)sample * nseg + g], len = seg_end[g] - seg_start[g] + 1;
		double* const out = rows + g * ld + col0 + sample;
		if(A == 0)
			*out = 0.0;                                         // no read: the sum is 0.0 and so is int(0.0) / 1000.0
		else {
			f = true;
			if(A < (1ull << 40)) {
				const uint64_t num = 1000ull * A, m = num / len, r = num - m * len;
				if(r != 0 && m < (1ull << 31)) {
					const uint64_t dist = (r < len - r)? r : len - r;
					const double bound = 2000.0 * (double)(A + 2) * (double)A * 1.1102230246251565e-16;   // 2 x 1000 (A + 1) u A, in units of 1 / len
					if(bound < (double)dist) {
						f = false;
						*out = __ddiv_rn((double)(int)m, 1000.0);
					}
				}
			}
		}
	}
	const uint32_t bits = __ballot_sync(FULL, f);
	if((threadIdx.x & 31) == 0 && g < nseg) {
		flag_bits[(uint64_t)sample * nwords + (g >> 5)] = bits;
		if(bits)
			atomicAdd(&nflagged[sample], (uint32_t)__popc(bits));
	}
}

// pass 2, tile filter: one thread per tile of the batch.  A tile whose window range holds no flagged window (reads in scaffold or coordinate order: a
// tile spans a few scaffolds, and most tiles stop here) gets a pair count of zero; the others are listed (in no particular order: every tile writes
// its pairs at its own offset).  ALL: every tile is listed.
__global__ void __launch_bounds__(256) k_cov_tile_filter(const ReadSrc* __restrict__ srcs, uint32_t ns, uint32_t total_tiles, const uint32_t* __restrict__ flag_bits,
                                                         uint32_t nwords, const uint32_t* __restrict__ nflagged, const uint2* __restrict__ tile_range, int all,
                                                         uint32_t* __restrict__ tile_counts, uint2* __restrict__ list, uint32_t* __restrict__ nlist)
{
	abw_grid_wait();
	const uint32_t flat = blockIdx.x * blockDim.x + threadIdx.x;
	bool go = false;
	uint32_t sample = 0;
	if(flat < total_tiles) {
		while(sample + 1 < ns && srcs[sample + 1].tile0 <= flat)
			sample++;
		go = all != 0;
		if(!all) {
			const uint2 tr = tile_range[flat];
			if(tr.x <= tr.y && nflagged[sample] > 0) {
				const uint32_t* __restrict__ flags = flag_bits + (uint64_t)sample * nwords;
				const uint32_t w0 = tr.x >> 5, w1 = tr.y >> 5;
				if(w1 - w0 >= 256u)
					go = true;                                  // reads in no particular order: the tile spans everything
				else
					for(uint32_t w = w0; w <= w1 && !go; w++) {
						uint32_t m = __ldg(flags + w);
						if(w == w0) m &= 0xFFFFFFFFu << (tr.x & 31u);
						if(w == w1) m &= 0xFFFFFFFFu >> (31u - (tr.y & 31u));
						go = m != 0;
					}
			}
			if(!go)
				tile_counts[flat] = 0;
		}
	}
	// warp-aggregated append
	const uint32_t m = __ballot_sync(FULL, go);
	if(m) {
		const int lane = threadIdx.x & 31;
		uint32_t base = 0;
		if(lane == __ffs(m) - 1)
			base = atomicAdd(nlist, (uint32_t)__popc(m));
		base = __shfl_sync(FULL, base, __ffs(m) - 1);
		if(go)
			list[base + __popc(m & ((1u << lane) - 1u))] = make_uint2(sample, flat - srcs[sample].tile0);
	}
}

// pass 2, count (EMIT = false) and emit (EMIT = true): the (window, overlap) pairs of the reads of a listed tile, in read order then window order, for the
// flagged windows only (ALL = false) or for every window (ALL = true).  key = sample * nseg + window.  CTAs walk the list.
template <bool EMIT, bool ALL>
__global__ void __launch_bounds__(COV_THREADS) k_cov_pairs(const ReadSrc* __restrict__ srcs, uint32_t max_snps, uint32_t nscaf, const uint4* __restrict__ scaf_info,
                                                          const uint64_t* __restrict__ seg_end, uint64_t nseg, const uint32_t* __restrict__ flag_bits, uint32_t nwords,
                                                          const uint2* __restrict__ list, const uint32_t* __restrict__ nlist, uint32_t* __restrict__ tile_counts,
                                                          const uint64_t* __restrict__ tile_offs, uint32_t* __restrict__ keys, uint32_t* __restrict__ vals,
                                                          unsigned long long* __restrict__ scaf_nbps, int nbps_sample)
{
	abw_grid_wait();
	__shared__ uint32_t sm[COV_THREADS / 32];
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	const uint32_t n = *nlist;
	for(uint32_t li = blockIdx.x; li < n; li += gridDim.x) {
		const uint2 ent = list[li];
		const uint32_t sample = ent.x, tile = ent.y;
		const ReadSrc src = srcs[sample];
		const uint32_t flat = src.tile0 + tile;
		const uint32_t* __restrict__ flags = ALL? nullptr : flag_bits + (uint64_t)sample * nwords;
		if(EMIT && tile_counts[flat] == 0)
			continue;                                           // uniform over the CTA
		const uint64_t r0 = ((uint64_t)tile * COV_THREADS + threadIdx.x) * COV_ITEMS;
		Rd4 rd;
		load_reads4(src, r0, max_snps, nscaf, rd);
		uint4 si[COV_ITEMS];
#pragma unroll
		for(int j = 0; j < COV_ITEMS; j++)
			si[j] = rd.acc[j]? __ldg(scaf_info + rd.scaf[j]) : make_uint4(0, 0, 1, 0);
		if(!EMIT && ALL && scaf_nbps != nullptr && (int)sample == nbps_sample) {
#pragma unroll
			for(int j = 0; j < COV_ITEMS; j++)
				warp_add_by_key(scaf_nbps, rd.scaf[j], rd.len[j], rd.acc[j]);
		}
		uint32_t c = 0;
#pragma unroll
		for(int j = 0; j < COV_ITEMS; j++) {
			if(!(rd.acc[j] && si[j].y > 0))
				continue;
			uint32_t g, o1, o2;
			if(regular_two(si[j], rd.pos0[j], rd.len[j], g, o1, o2)) {
				if(o1 && (ALL || ((__ldg(flags + (g >> 5)) >> (g & 31u)) & 1u)))
					c++;
				if(o2 && (ALL || ((__ldg(flags + ((g + 1u) >> 5)) >> ((g + 1u) & 31u)) & 1u)))
					c++;
				continue;
			}
			WinIter it;
			it.init(rd.pos0[j], rd.len[j], si[j], seg_end);
			for(; it.valid(); it.next())
				if(ALL || ((__ldg(flags + (it.g >> 5)) >> (it.g & 31u)) & 1u))
					c++;
		}
		if(!EMIT) {
			c = __reduce_add_sync(FULL, c);
			if(lane == 0)
				sm[warp] = c;
			__syncthreads();
			if(threadIdx.x == 0) {
				uint32_t t = 0;
#pragma unroll
				for(int w = 0; w < COV_THREADS / 32; w++)
					t += sm[w];
				tile_counts[flat] = t;
			}
			__syncthreads();
			continue;
		}
		uint32_t incl = c;
#pragma unroll
		for(int o = 1; o < 32; o <<= 1) {
			const uint32_t t = __shfl_up_sync(FULL, incl, o);
			if(lane >= o)
				incl += t;
		}
		if(lane == 31)
			sm[warp] = incl;
		__syncthreads();
		uint32_t wex = 0;
#pragma unroll
		for(int w = 0; w < COV_THREADS / 32; w++)
			if(w < warp)
				wex += sm[w];
		__syncthreads();
		if(c == 0)
			continue;
		uint64_t o = tile_offs[flat] + wex + incl - c;
		const uint32_t key0 = (uint32_t)((uint64_t)sample * nseg);
#pragma unroll
		for(int j = 0; j < COV_ITEMS; j++) {
			if(!(rd.acc[j] && si[j].y > 0))
				continue;
			uint32_t g, o1, o2;
			if(regular_two(si[j], rd.pos0[j], rd.len[j], g, o1, o2)) {
				if(o1 && (ALL || ((__ldg(flags + (g >> 5)) >> (g & 31u)) & 1u))) {
					keys[o] = key0 + g;
					vals[o] = o1;
					o++;
				}
				if(o2 && (ALL || ((__ldg(flags + ((g + 1u) >> 5)) >> ((g + 1u) & 31u)) & 1u))) {
					keys[o] = key0 + g + 1u;
					vals[o] = o2;
					o++;
				}
				continue;
			}
			WinIter it;
			it.init(rd.pos0[j], rd.len[j], si[j], seg_end);
			for(; it.valid(); it.next())
				if(ALL || ((__ldg(flags + (it.g >> 5)) >> (it.g & 31u)) & 1u)) {
					keys[o] = key0 + it.g;
					vals[o] = it.overlap();                     // the overlap travels with the pair: no gather after the sort
					o++;
				}
		}
	}
}

// The pairs were sorted stably by (sample, window): the thread at the first pair of a window adds its reads in SAM order (quirk Q5) with exactly the
// reference's operations, BATCH loads in flight.  Windows without a pair keep what k_cov_quotient (or the zero fill) left.
template <int KIND, int BATCH>
__global__ void __launch_bounds__(128) k_cov_accumulate(const uint32_t* __restrict__ keys, const uint32_t* __restrict__ vals, uint64_t npairs, uint64_t nseg,
                                                        const uint64_t* __restrict__ seg_start, const uint64_t* __restrict__ seg_end, double* __restrict__ rows,
                                                        uint64_t ld, uint32_t col0)
{
	abw_grid_wait();
	const uint64_t i0 = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if(i0 >= npairs)
		return;
	const uint32_t key = keys[i0];
	if(i0 > 0 && keys[i0 - 1] == key)
		return;
	const uint32_t sample = (uint32_t)(key / nseg);
	const uint64_t g = key - (uint64_t)sample * nseg;
	const double seglen = (double)(seg_end[g] - seg_start[g] + 1);
	double acc = 0.0, q = 0.0;
	uint32_t last = 0xFFFFFFFFu;
	bool more = true;
	for(uint64_t i = i0; more && i < npairs; i += BATCH) {
		uint32_t kk[BATCH], ov[BATCH];
#pragma unroll
		for(int j = 0; j < BATCH; j++) {
			const bool in = i + j < npairs;
			kk[j] = in? __ldg(keys + i + j) : ~key;
			ov[j] = in? __ldg(vals + i + j) : 0u;
		}
#pragma unroll
		for(int j = 0; j < BATCH; j++) {
			if(more && kk[j] == key) {
				if(ov[j] != last) {                             // most reads lie entirely inside the window: same quotient, computed once
					q = __ddiv_rn((double)ov[j], seglen);       // :184
					last = ov[j];
				}
				acc = __dadd_rn(acc, q);
			}
			else
				more = false;
		}
	}
	if(KIND == ABW_FEAT_TRUNC3)
		acc = __ddiv_rn((double)__double2int_rz(__dmul_rn(1000.0, acc)), 1000.0);
	rows[g * ld + col0 + sample] = acc;
}

__global__ void k_cov_zero_columns(double* __restrict__ rows, uint64_t nseg, uint64_t ld, uint32_t col0, uint32_t ncols)
{
	abw_grid_wait();
	const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if(i < nseg * ncols)
		rows[(i / ncols) * ld + col0 + (i % ncols)] = 0.0;
}

// pass 2 for the samples [0, ns) of a group whose ReadSrc records are at d_srcs
int coverage_pairs(abw_ctx* ctx, const abw_segments* g, const ReadSrc* d_srcs, uint32_t ns, uint32_t total_tiles, uint32_t max_snps, int kind,
                   double* d_rows, uint64_t ld, uint32_t col0, bool all, const uint32_t* flags, uint32_t nwords, const uint32_t* nflagged, const uint2* tile_range,
                   unsigned long long* d_scaf_nbps, int nbps_sample)
{
	if(total_tiles == 0 || g->nseg == 0)
		return ABW_OK;
	DevBuf<uint32_t> tile_counts, keys, keys_tmp, vals, vals_tmp, nlist;
	DevBuf<uint64_t> tile_offs, total;
	DevBuf<uint2> list;
	ABW_CUDA(ctx, tile_counts.alloc(total_tiles));
	ABW_CUDA(ctx, tile_offs.alloc(total_tiles));
	ABW_CUDA(ctx, total.alloc(1));
	ABW_CUDA(ctx, list.alloc(total_tiles));
	ABW_CUDA(ctx, nlist.alloc(1));
	ABW_CUDA(ctx, cudaMemsetAsync(nlist.p, 0, sizeof(uint32_t), ctx->stream));
	ABW_LAUNCH(ctx, k_cov_tile_filter, abw_div_up(total_tiles, 256), 256, 0, d_srcs, ns, total_tiles, flags, nwords, nflagged, tile_range, all? 1 : 0, tile_counts.p, list.p,
	           nlist.p);
	const unsigned int grid = std::min<unsigned int>(total_tiles, 8u * (unsigned)ctx->sm_count);
	if(all)
		ABW_LAUNCH(ctx, (k_cov_pairs<false, true>), grid, COV_THREADS, 0, d_srcs, max_snps, g->nscaf, g->scaf_info.p, g->seg_end.p, g->nseg, flags, nwords,
		           (const uint2*)list.p, (const uint32_t*)nlist.p, tile_counts.p, (const uint64_t*)nullptr, (uint32_t*)nullptr, (uint32_t*)nullptr, d_scaf_nbps, nbps_sample);
	else
		ABW_LAUNCH(ctx, (k_cov_pairs<false, false>), grid, COV_THREADS, 0, d_srcs, max_snps, g->nscaf, g->scaf_info.p, g->seg_end.p, g->nseg, flags, nwords,
		           (const uint2*)list.p, (const uint32_t*)nlist.p, tile_counts.p, (const uint64_t*)nullptr, (uint32_t*)nullptr, (uint32_t*)nullptr,
		           (unsigned long long*)nullptr, -1);
	ABW_CHECK(abw_exclusive_scan_u32_to_u64(ctx, tile_counts.p, tile_offs.p, total_tiles, total.p));
	uint64_t npairs = 0;
	ABW_CUDA(ctx, abw_fetch(ctx, &npairs, total.p, sizeof(uint64_t)));
	ABW_CUDA(ctx, abw_sync(ctx));
	if(npairs == 0)
		return ABW_OK;
	if(npairs >= (1ull << 32))
		return abw_fail(ctx, ABW_ERR_UNSUPPORTED, "abw_coverage: more than 2^32-1 (window, read) pairs per call; split the samples");
	ABW_CUDA(ctx, keys.alloc(npairs));
	ABW_CUDA(ctx, keys_tmp.alloc(npairs));
	ABW_CUDA(ctx, vals.alloc(npairs));
	ABW_CUDA(ctx, vals_tmp.alloc(npairs));
	if(all)
		ABW_LAUNCH(ctx, (k_cov_pairs<true, true>), grid, COV_THREADS, 0, d_srcs, max_snps, g->nscaf, g->scaf_info.p, g->seg_end.p, g->nseg, flags, nwords,
		           (const uint2*)list.p, (const uint32_t*)nlist.p, tile_counts.p, (const uint64_t*)tile_offs.p, keys.p, vals.p, (unsigned long long*)nullptr, -1);
	else
		ABW_LAUNCH(ctx, (k_cov_pairs<true, false>), grid, COV_THREADS, 0, d_srcs, max_snps, g->nscaf, g->scaf_info.p, g->seg_end.p, g->nseg, flags, nwords,
		           (const uint2*)list.p, (const uint32_t*)nlist.p, tile_counts.p, (const uint64_t*)tile_offs.p, keys.p, vals.p, (unsigned long long*)nullptr, -1);
	int nbits = 1;
	while(nbits < 32 && (1ull << nbits) < (uint64_t)ns * g->nseg)
		nbits++;
	// (sample, window) ids are dense: every bit below nbits is taken as varying, no inspection pass
	ABW_CHECK(abw_radix_sort_pairs_u32(ctx, keys.p, keys_tmp.p, vals.p, vals_tmp.p, npairs, 1, npairs, -nbits));
	const unsigned int blocks = abw_div_up(npairs, 128);
	if(kind == ABW_FEAT_TRUNC3)
		ABW_LAUNCH(ctx, (k_cov_accumulate<ABW_FEAT_TRUNC3, 16>), blocks, 128, 0, keys.p, vals.p, npairs, g->nseg, g->seg_start.p, g->seg_end.p, d_rows, ld, col0);
	else
		ABW_LAUNCH(ctx, (k_cov_accumulate<ABW_FEAT_RAW, 8>), blocks, 128, 0, keys.p, vals.p, npairs, g->nseg, g->seg_start.p, g->seg_end.p, d_rows, ld, col0);
	return ABW_OK;
}

int coverage_batch(abw_ctx* ctx, const abw_segments* g, const abw_sample* samples, uint32_t nsamples, uint32_t max_snps, int kind, double* d_rows, uint64_t ld,
                   uint32_t col0, int32_t this_sample, uint64_t* d_scaf_nbps)
{
	if(nsamples == 0 || g->nseg == 0)
		return ABW_OK;
	const bool all = (kind == ABW_FEAT_RAW);
	const uint32_t nwords = (uint32_t)((g->nseg + 31) / 32);
	// samples are processed in groups: (sample, window) keys must fit 32 bits and the integer sums a few GB
	const uint64_t by_key = std::max<uint64_t>(1, ((1ull << 32) - 1) / g->nseg), by_mem = std::max<uint64_t>(1, (4ull << 30) / (8 * g->nseg));
	const uint32_t group = (uint32_t)std::min<uint64_t>(std::min(by_key, by_mem), nsamples);
	for(uint32_t s0 = 0; s0 < nsamples; s0 += group) {
		const uint32_t ns = std::min(group, nsamples - s0);
		std::vector<ReadSrc> srcs(ns);
		// sorted samples are decoded into compact records, which pass 2 reads again: they live until the end of the group
		std::vector<DevBuf<abw_read8>> decoded(ns);
		uint32_t total_tiles = 0;
		for(uint32_t j = 0; j < ns; j++) {
			const abw_sample& sm = samples[s0 + j];
			ReadSrc& r = srcs[j];
			r.p = sm.reads; r.n = sm.nreads; r.len16 = sm.len16; r.len = sm.len; r.fmt = sm.format;
			if(sm.format == ABW_READS_SORTED) {
				ABW_CUDA(ctx, decoded[j].alloc(sm.nreads));
				r.p = decoded[j].p;
				r.fmt = ABW_READS_COMPACT;
			}
			r.tile0 = total_tiles;
			r.ntiles = abw_div_up(sm.nreads, COV_TILE);
			total_tiles += r.ntiles;
		}
		DevBuf<ReadSrc> d_srcs;
		DevBuf<unsigned long long> sum_ov;
		DevBuf<uint32_t> flags, nflagged;
		DevBuf<uint2> tile_range;
		ABW_CUDA(ctx, d_srcs.alloc(ns));
		ABW_CUDA(ctx, abw_upload_small(ctx, d_srcs.p, srcs.data(), sizeof(ReadSrc) * ns));
		const int nbps_local = (this_sample >= (int32_t)s0 && this_sample < (int32_t)(s0 + ns) && d_scaf_nbps)? (int)(this_sample - (int32_t)s0) : -1;
		if(all) {
			for(uint32_t j = 0; j < ns; j++)
				ABW_CHECK(abw_wait_h2d(ctx, samples[s0 + j].h2d_ticket));
			for(uint32_t j = 0; j < ns; j++)
				if(samples[s0 + j].format == ABW_READS_SORTED)
					ABW_CHECK(abw_decode_sorted_reads(ctx, samples[s0 + j], decoded[j].p));
			ABW_LAUNCH(ctx, k_cov_zero_columns, abw_div_up(g->nseg * ns, 256), 256, 0, d_rows, g->nseg, ld, col0 + s0, ns);
			ABW_CHECK(coverage_pairs(ctx, g, d_srcs.p, ns, total_tiles, max_snps, kind, d_rows, ld, col0 + s0, true, nullptr, nwords, nullptr, nullptr,
			                         (unsigned long long*)d_scaf_nbps, nbps_local));
			continue;
		}
		ABW_CUDA(ctx, sum_ov.alloc((size_t)ns * g->nseg));
		ABW_CUDA(ctx, flags.alloc((size_t)ns * nwords));
		ABW_CUDA(ctx, nflagged.alloc(ns));
		ABW_CUDA(ctx, tile_range.alloc(std::max<uint32_t>(total_tiles, 1)));
		ABW_CUDA(ctx, cudaMemsetAsync(sum_ov.p, 0, sizeof(unsigned long long) * ns * g->nseg, ctx->stream));
		ABW_CUDA(ctx, cudaMemsetAsync(nflagged.p, 0, sizeof(uint32_t) * ns, ctx->stream));
		for(uint32_t j = 0; j < ns; j++) {
			ABW_CHECK(abw_wait_h2d(ctx, samples[s0 + j].h2d_ticket));           // the sample's records may still be on their way (abw_h2d_async)
			if(samples[s0 + j].format == ABW_READS_SORTED)
				ABW_CHECK(abw_decode_sorted_reads(ctx, samples[s0 + j], decoded[j].p));
			if(srcs[j].ntiles == 0)
				continue;
			if((int)j == nbps_local)
				ABW_LAUNCH(ctx, k_cov_sum<true>, srcs[j].ntiles, COV_THREADS, 0, srcs[j], max_snps, g->nscaf, g->scaf_info.p, g->seg_end.p, sum_ov.p + (size_t)j * g->nseg,
				           tile_range.p, (unsigned long long*)d_scaf_nbps);
			else
				ABW_LAUNCH(ctx, k_cov_sum<false>, srcs[j].ntiles, COV_THREADS, 0, srcs[j], max_snps, g->nscaf, g->scaf_info.p, g->seg_end.p, sum_ov.p + (size_t)j * g->nseg,
				           tile_range.p, (unsigned long long*)nullptr);
		}
		ABW_LAUNCH(ctx, k_cov_quotient, dim3(abw_div_up(g->nseg, 256), ns), 256, 0, sum_ov.p, g->nseg, g->seg_start.p, g->seg_end.p, d_rows, ld, col0 + s0, flags.p, nwords,
		           nflagged.p);
		ABW_CHECK(coverage_pairs(ctx, g, d_srcs.p, ns, total_tiles, max_snps, kind, d_rows, ld, col0 + s0, false, flags.p, nwords, nflagged.p, tile_range.p,
		                         nullptr, -1));
	}
	return ABW_OK;
}

}  // namespace

extern "C" {

int abw_coverage_batch(abw_ctx* ctx, const abw_segments* g, const abw_sample* h_samples, uint32_t nsamples, uint32_t max_snps, int kind, double* d_rows, uint64_t ld,
                       uint32_t col0, int32_t this_sample, uint64_t* d_scaf_nbps)
{
	if(!ctx || !g || !d_rows || (!h_samples && nsamples))
		return abw_fail(ctx, ABW_ERR_ARG, "abw_coverage_batch: null argument");
	if(kind != ABW_FEAT_TRUNC3 && kind != ABW_FEAT_RAW)
		return abw_fail(ctx, ABW_ERR_ARG, "abw_coverage_batch: unknown kind");
	if(ld < (uint64_t)col0 + nsamples)
		return abw_fail(ctx, ABW_ERR_ARG, "abw_coverage_batch: row stride too small");
	if(g->nseg >= (1ull << 32))
		return abw_fail(ctx, ABW_ERR_UNSUPPORTED, "abw_coverage: more than 2^32-1 windows");
	for(uint32_t j = 0; j < nsamples; j++) {
		const abw_sample& sm = h_samples[j];
		if(!sm.reads && sm.nreads)
			return abw_fail(ctx, ABW_ERR_ARG, "abw_coverage_batch: null read records");
		if(sm.format != ABW_READS_FULL && sm.format != ABW_READS_COMPACT && sm.format != ABW_READS_SORTED)
			return abw_fail(ctx, ABW_ERR_ARG, "abw_coverage_batch: unknown record format");
		if(sm.format == ABW_READS_SORTED) {
			if((!sm.runs && sm.nruns) || (!sm.exc && sm.nexc))
				return abw_fail(ctx, ABW_ERR_ARG, "abw_coverage_batch: null runs or escape array");
			if(sm.nexc > sm.nreads)
				return abw_fail(ctx, ABW_ERR_ARG, "abw_coverage_batch: more escapes than reads");
			if(sm.nruns >= (1ull << 32))
				return abw_fail(ctx, ABW_ERR_ARG, "abw_coverage_batch: 2^32 runs or more");
		}
		if(sm.nreads >= (1ull << 32))
			return abw_fail(ctx, ABW_ERR_UNSUPPORTED, "abw_coverage: more than 2^32-1 reads per sample; split the sample");
	}
	ABW_ENTER(ctx);
	return coverage_batch(ctx, g, h_samples, nsamples, max_snps, kind, d_rows, ld, col0, this_sample, d_scaf_nbps);
}

int abw_coverage(abw_ctx* ctx, const abw_segments* g, const abw_read* reads, uint64_t nreads, int reads_on_device, uint32_t max_snps,
                 int kind, double* d_rows, uint64_t ld, uint32_t col, uint64_t* d_scaf_nbps)
{
	if(!ctx || !g || !d_rows || (!reads && nreads))
		return abw_fail(ctx, ABW_ERR_ARG, "abw_coverage: null argument");
	if(nreads >= (1ull << 32))
		return abw_fail(ctx, ABW_ERR_UNSUPPORTED, "abw_coverage: more than 2^32-1 reads per call; split the sample");
	if(g->nseg >= (1ull << 32))
		return abw_fail(ctx, ABW_ERR_UNSUPPORTED, "abw_coverage: more than 2^32-1 windows");
	if(kind != ABW_FEAT_TRUNC3 && kind != ABW_FEAT_RAW)
		return abw_fail(ctx, ABW_ERR_ARG, "abw_coverage: unknown kind");
	ABW_ENTER(ctx);
	DevBuf<abw_read> d_reads;
	abw_sample sm{};
	sm.reads = reads; sm.nreads = nreads; sm.format = ABW_READS_FULL; sm.len = 0; sm.len16 = nullptr; sm.h2d_ticket = 0;
	if(!reads_on_device && nreads) {
		ABW_CUDA(ctx, d_reads.alloc(nreads));
		ABW_CUDA(ctx, cudaMemcpyAsync(d_reads.p, reads, sizeof(abw_read) * nreads, cudaMemcpyHostToDevice, ctx->stream));
		sm.reads = d_reads.p;
	}
	ABW_CHECK(coverage_batch(ctx, g, &sm, 1, max_snps, kind, d_rows, ld, col, d_scaf_nbps? 0 : -1, d_scaf_nbps));
	// results stay on the device and every later entry point works in the order of the context stream: only a host buffer of reads has to be
	// released by the time the call returns
	if(!reads_on_device)
		ABW_CUDA(ctx, abw_sync(ctx));
	return ABW_OK;
}

}  // extern "C"
