// ABW_READS_SORTED -> abw_read8: the decode of coordinate-sorted read records (include/abawaca_b200.h, DESIGN.md section 4) on the device.
//
// pos0 of read i is a linear recurrence over the reads in order: pos[i] = E(k) at an escape (k = escapes before i), delta[i] at the first read of a
// run, pos[i-1] + delta[i] otherwise.  That is a segmented prefix sum of the deltas which restarts at run starts and at escapes; its elements are
// (restarts, value) with (f1, v1) . (f2, v2) = f2? (f2, v2) : (f1, v1 + v2), all 32-bit arithmetic.  The value an escape restarts with needs the
// GLOBAL escape count k, so the decode of a sample runs in tiles of RC_TILE reads:
//   k_sorted_run_counts  the run counts as a uint32 array, whose exclusive scan (abw_exclusive_scan_u32_to_u64) gives the first read of every run
//   k_sorted_tile_runs   one thread per tile: the run of the tile's first read (binary search)
//   k_sorted_summary     per tile: escapes in it, and its segmented summary with the value of its last restart left symbolic (an escape's local
//                        index or "run start")
//   k_sorted_carry       one CTA: scans the escape counts (every tile's exc base), resolves the symbolic restarts with exc[], and scans the tile
//                        summaries (every tile's carry-in: pos0 of the read before it)
//   k_sorted_write       per tile: the same restarts again, scanned inside the tile from the carry-in, and 8-byte records out
// The run of a read is found by binary search in the run starts, between the runs of its tile's first read and of the next tile's first read.  Skipped reads get scaf 0xFFFFFFFF, which every
// coverage kernel treats as an unknown scaffold.
#include "features.cuh"

namespace {

constexpr uint32_t FULL = 0xffffffffu;
constexpr int RC_THREADS = 256;
constexpr int RC_ITEMS = 8;                                 // consecutive reads per thread: one 16-byte load of deltas
constexpr int RC_TILE = RC_THREADS * RC_ITEMS;
constexpr int RC_CARRY_THREADS = 512;
constexpr int RC_CARRY_TILES = 4;                          // consecutive tiles per thread of k_sorted_carry
constexpr uint32_t RC_ESC = 0xFFFFu;
constexpr uint32_t RC_SKIP = 0xFFFFFFFFu;

struct Seg {
	uint32_t f, v;                                          // f: the range restarts the sum; v: value after the range (f) or sum of its deltas (!f)
};
__device__ __forceinline__ Seg seg_op(Seg a, Seg b) { return b.f? b : Seg{a.f, a.v + b.v}; }

// exclusive scan of one element per thread across the CTA, `carry` in front of thread 0; *total (every thread) = carry . all.  sm: NT / 32 entries.
// A plain sum is the scan of elements with f = 0.
template <int NT>
__device__ __forceinline__ Seg block_seg_scan(Seg x, Seg carry, Seg* total, Seg* sm)
{
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	Seg incl = x;
#pragma unroll
	for(int o = 1; o < 32; o <<= 1) {
		const Seg y{__shfl_up_sync(FULL, incl.f, o), __shfl_up_sync(FULL, incl.v, o)};
		if(lane >= o)
			incl = seg_op(y, incl);
	}
	if(lane == 31)
		sm[warp] = incl;
	__syncthreads();
	Seg pre = carry;
	for(int w = 0; w < warp; w++)
		pre = seg_op(pre, sm[w]);
	Seg all = pre;
	for(int w = warp; w < NT / 32; w++)
		all = seg_op(all, sm[w]);
	*total = all;
	const Seg up{__shfl_up_sync(FULL, incl.f, 1), __shfl_up_sync(FULL, incl.v, 1)};
	__syncthreads();
	return lane? seg_op(pre, up) : pre;
}

__global__ void __launch_bounds__(256) k_sorted_run_counts(const abw_read_run* __restrict__ runs, uint64_t nruns, uint32_t* __restrict__ counts)
{
	abw_grid_wait();
	const uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if(r < nruns)
		counts[r] = __ldg(&runs[r].count);
}

// last run r in [lo, hi) with first[r] <= i, given first[lo] <= i
__device__ __forceinline__ uint32_t run_search(const uint64_t* __restrict__ first, uint32_t lo, uint32_t hi, uint64_t i)
{
	while(hi - lo > 1) {
		const uint32_t mid = lo + ((hi - lo) >> 1);
		if(__ldg(first + mid) <= i) lo = mid; else hi = mid;
	}
	return lo;
}

// tile_run[t] = run of read t * RC_TILE, nruns when that read has no run.  A launch of its own: the dependent loads of the search are paid once per
// tile in parallel, not at the start of every CTA of the decode kernels.
__global__ void __launch_bounds__(256) k_sorted_tile_runs(const uint64_t* __restrict__ first, uint32_t nruns, const uint64_t* __restrict__ d_total, uint64_t n,
                                                          uint32_t ntiles, uint32_t* __restrict__ tile_run)
{
	abw_grid_wait();
	const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
	if(t >= ntiles)
		return;
	const uint64_t i = (uint64_t)t * RC_TILE;
	tile_run[t] = (nruns && i < min(n, *d_total))? run_search(first, 0, nruns, i) : nruns;
}

// The RC_ITEMS reads of this thread: deltas, and per read its run (nruns: none, the read lies past the sum of the counts) and whether it starts one.
// Every search lies between the run of the tile's first read and that of the next tile's first read (a step or two when runs are long).
struct Items {
	uint32_t d[RC_ITEMS];
	uint32_t run[RC_ITEMS];
	bool     start[RC_ITEMS];
};

__device__ __forceinline__ void load_items(const uint16_t* __restrict__ delta, uint64_t n, const uint64_t* __restrict__ first, uint32_t nruns, uint64_t total,
                                           const uint32_t* __restrict__ tile_run, uint32_t ntiles, Items& it)
{
	const uint64_t tile = blockIdx.x, i0 = tile * RC_TILE + (uint64_t)threadIdx.x * RC_ITEMS;
	const uint32_t lo = __ldg(tile_run + tile), nx = (tile + 1 < ntiles)? __ldg(tile_run + tile + 1) : nruns;
	const uint32_t hi = (nx < nruns)? nx + 1 : nruns;
	if(i0 + RC_ITEMS <= n && (reinterpret_cast<uintptr_t>(delta + i0) & 15u) == 0) {
		const uint4 a = __ldg(reinterpret_cast<const uint4*>(delta + i0));
		const uint32_t w[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
		for(int j = 0; j < RC_ITEMS; j++)
			it.d[j] = (w[j >> 1] >> (16 * (j & 1))) & 0xFFFFu;
	}
	else {
#pragma unroll
		for(int j = 0; j < RC_ITEMS; j++)
			it.d[j] = (i0 + j < n)? (uint32_t)__ldg(delta + i0 + j) : 0u;
	}
	uint32_t r = (i0 < total && nruns)? run_search(first, lo, hi, i0) : 0;
#pragma unroll
	for(int j = 0; j < RC_ITEMS; j++) {
		const uint64_t i = i0 + j;
		if(i >= total || nruns == 0) {
			it.run[j] = nruns;
			it.start[j] = false;
			continue;
		}
		if(r + 1 < hi && __ldg(first + r + 1) <= i)
			r = run_search(first, r + 1, hi, i);
		it.run[j] = r;
		it.start[j] = __ldg(first + r) == i;
	}
}

// per tile: {escapes, restart code, escapes before the last restart, sum of the deltas from the last restart on}.  Restart code: 0 none, else
// (index in the tile + 1) * 2 + (the restart is an escape); the largest code is the last restart.
__global__ void __launch_bounds__(RC_THREADS) k_sorted_summary(const uint16_t* __restrict__ delta, uint64_t n, const uint64_t* __restrict__ first, uint32_t nruns,
                                                               const uint64_t* __restrict__ d_total, const uint32_t* __restrict__ tile_run, uint32_t ntiles,
                                                               uint4* __restrict__ summary)
{
	abw_grid_wait();
	__shared__ uint32_t sm_esc, sm_code, sm_before, sm_add;
	if(threadIdx.x == 0) {
		sm_esc = 0; sm_code = 0; sm_before = 0; sm_add = 0;
	}
	__syncthreads();
	Items it;
	load_items(delta, n, first, nruns, nruns? *d_total : 0, tile_run, ntiles, it);
	const uint32_t base = threadIdx.x * RC_ITEMS;
	uint32_t esc = 0, code = 0;
#pragma unroll
	for(int j = 0; j < RC_ITEMS; j++) {
		const bool in = (uint64_t)blockIdx.x * RC_TILE + base + j < n;
		const bool e = in && it.d[j] == RC_ESC;
		esc += e;
		if(in && (e || it.start[j]))
			code = (base + j + 1) * 2 + (e? 1u : 0u);
	}
	esc = __reduce_add_sync(FULL, esc);
	code = __reduce_max_sync(FULL, code);
	if((threadIdx.x & 31) == 0) {
		atomicAdd(&sm_esc, esc);
		atomicMax(&sm_code, code);
	}
	__syncthreads();
	const uint32_t c = sm_code, rst = c? c / 2 - 1 : 0;
	uint32_t before = 0, add = 0;
#pragma unroll
	for(int j = 0; j < RC_ITEMS; j++) {
		const bool in = (uint64_t)blockIdx.x * RC_TILE + base + j < n;
		const bool e = in && it.d[j] == RC_ESC;
		if(e && base + j < rst)
			before++;
		if(in && !e && base + j >= rst)
			add += it.d[j];
	}
	before = __reduce_add_sync(FULL, before);
	add = __reduce_add_sync(FULL, add);
	if((threadIdx.x & 31) == 0) {
		atomicAdd(&sm_before, before);
		atomicAdd(&sm_add, add);
	}
	__syncthreads();
	if(threadIdx.x == 0)
		summary[blockIdx.x] = make_uint4(sm_esc, c, sm_before, sm_add);
}

__device__ __forceinline__ uint32_t exc_at(const uint32_t* __restrict__ exc, uint64_t nexc, uint64_t k) { return k < nexc? __ldg(exc + k) : 0u; }

// one CTA: per tile {escapes before it, pos0 of the read before it}; RC_CARRY_TILES consecutive tiles per thread
__global__ void __launch_bounds__(RC_CARRY_THREADS) k_sorted_carry(const uint4* __restrict__ summary, uint32_t ntiles, const uint32_t* __restrict__ exc, uint64_t nexc,
                                                                   uint2* __restrict__ carry)
{
	abw_grid_wait();
	__shared__ Seg sm[RC_CARRY_THREADS / 32];
	Seg esc_carry{0, 0}, pos_carry{0, 0};
	for(uint32_t c0 = 0; c0 < ntiles; c0 += RC_CARRY_THREADS * RC_CARRY_TILES) {
		const uint32_t t0 = c0 + threadIdx.x * RC_CARRY_TILES;
		uint4 s[RC_CARRY_TILES];
		uint32_t esc = 0;
#pragma unroll
		for(int q = 0; q < RC_CARRY_TILES; q++) {
			s[q] = (t0 + q < ntiles)? summary[t0 + q] : make_uint4(0, 0, 0, 0);
			esc += s[q].x;
		}
		Seg tot;
		const uint32_t kbase = block_seg_scan<RC_CARRY_THREADS>(Seg{0, esc}, esc_carry, &tot, sm).v;
		esc_carry = tot;
		Seg e[RC_CARRY_TILES], x{0, 0};
		uint32_t k = kbase;
#pragma unroll
		for(int q = 0; q < RC_CARRY_TILES; q++) {
			e[q] = Seg{s[q].y != 0, s[q].w};
			if(s[q].y & 1u)
				e[q].v += exc_at(exc, nexc, (uint64_t)k + s[q].z);
			k += s[q].x;
			x = seg_op(x, e[q]);
		}
		Seg pre = block_seg_scan<RC_CARRY_THREADS>(x, pos_carry, &tot, sm);
		pos_carry = tot;
		k = kbase;
#pragma unroll
		for(int q = 0; q < RC_CARRY_TILES; q++) {
			if(t0 + q < ntiles)
				carry[t0 + q] = make_uint2(k, pre.v);
			pre = seg_op(pre, e[q]);
			k += s[q].x;
		}
	}
}

__global__ void __launch_bounds__(RC_THREADS, 4) k_sorted_write(const uint16_t* __restrict__ delta, uint64_t n, const uint64_t* __restrict__ first, uint32_t nruns,
                                                             const uint64_t* __restrict__ d_total, const abw_read_run* __restrict__ runs, const uint32_t* __restrict__ exc,
                                                             uint64_t nexc, const uint32_t* __restrict__ tile_run, uint32_t ntiles, const uint2* __restrict__ carry,
                                                             abw_read8* __restrict__ out)
{
	abw_grid_wait();
	__shared__ Seg sm[RC_THREADS / 32];
	Items it;
	load_items(delta, n, first, nruns, nruns? *d_total : 0, tile_run, ntiles, it);
	const uint64_t i0 = (uint64_t)blockIdx.x * RC_TILE + (uint64_t)threadIdx.x * RC_ITEMS;
	const uint2 c = carry[blockIdx.x];
	uint32_t esc = 0;
#pragma unroll
	for(int j = 0; j < RC_ITEMS; j++)
		esc += (i0 + j < n && it.d[j] == RC_ESC);
	Seg tot;
	const uint64_t k0 = c.x + block_seg_scan<RC_THREADS>(Seg{0, esc}, Seg{0, 0}, &tot, sm).v;
	// this thread's segmented summary, then the pos0 of the read before its first one
	Seg x{0, 0};
	uint64_t k = k0;
#pragma unroll
	for(int j = 0; j < RC_ITEMS; j++) {
		if(i0 + j >= n)
			break;
		if(it.d[j] == RC_ESC)
			x = Seg{1, exc_at(exc, nexc, k++)};
		else if(it.start[j])
			x = Seg{1, it.d[j]};
		else
			x.v += it.d[j];
	}
	uint32_t pos = block_seg_scan<RC_THREADS>(x, Seg{0, c.y}, &tot, sm).v;
	uint2 rec[RC_ITEMS];
	k = k0;
#pragma unroll
	for(int j = 0; j < RC_ITEMS; j++) {
		bool keep = it.run[j] < nruns;
		if(it.d[j] == RC_ESC) {
			keep = keep && k < nexc;
			pos = exc_at(exc, nexc, k++);
		}
		else
			pos = (it.start[j]? 0u : pos) + it.d[j];
		rec[j] = make_uint2(keep? __ldg(&runs[it.run[j]].scaf) : RC_SKIP, pos);
	}
	uint2* __restrict__ o = reinterpret_cast<uint2*>(out);
	if(i0 + RC_ITEMS <= n && (reinterpret_cast<uintptr_t>(o + i0) & 15u) == 0) {
#pragma unroll
		for(int j = 0; j < RC_ITEMS; j += 2)
			*reinterpret_cast<uint4*>(o + i0 + j) = make_uint4(rec[j].x, rec[j].y, rec[j + 1].x, rec[j + 1].y);
	}
	else {
#pragma unroll
		for(int j = 0; j < RC_ITEMS; j++)
			if(i0 + j < n)
				o[i0 + j] = rec[j];
	}
}

}  // namespace

int abw_decode_sorted_reads(abw_ctx* ctx, const abw_sample& sm, abw_read8* d_out)
{
	const uint64_t n = sm.nreads, nruns = sm.nruns;
	if(n == 0)
		return ABW_OK;
	const uint32_t ntiles = abw_div_up(n, RC_TILE);
	DevBuf<uint32_t> counts, tile_run;
	DevBuf<uint64_t> first;
	DevBuf<uint4> summary;
	DevBuf<uint2> carry;
	ABW_CUDA(ctx, counts.alloc(nruns));
	ABW_CUDA(ctx, first.alloc(nruns + 1));                  // [nruns]: the sum of the counts
	ABW_CUDA(ctx, tile_run.alloc(ntiles));
	ABW_CUDA(ctx, summary.alloc(ntiles));
	ABW_CUDA(ctx, carry.alloc(ntiles));
	if(nruns) {
		ABW_LAUNCH(ctx, k_sorted_run_counts, abw_div_up(nruns, 256), 256, 0, sm.runs, nruns, counts.p);
		ABW_CHECK(abw_exclusive_scan_u32_to_u64(ctx, counts.p, first.p, nruns, first.p + nruns));
	}
	const uint16_t* delta = static_cast<const uint16_t*>(sm.reads);
	const uint64_t* total = first.p + nruns;
	ABW_LAUNCH(ctx, k_sorted_tile_runs, abw_div_up(ntiles, 256), 256, 0, (const uint64_t*)first.p, (uint32_t)nruns, total, n, ntiles, tile_run.p);
	ABW_LAUNCH(ctx, k_sorted_summary, ntiles, RC_THREADS, 0, delta, n, (const uint64_t*)first.p, (uint32_t)nruns, total, (const uint32_t*)tile_run.p, ntiles, summary.p);
	ABW_LAUNCH(ctx, k_sorted_carry, 1, RC_CARRY_THREADS, 0, (const uint4*)summary.p, ntiles, sm.exc, sm.nexc, carry.p);
	ABW_LAUNCH(ctx, k_sorted_write, ntiles, RC_THREADS, 0, delta, n, (const uint64_t*)first.p, (uint32_t)nruns, total, sm.runs, sm.exc, sm.nexc,
	           (const uint32_t*)tile_run.p, ntiles, (const uint2*)carry.p, d_out);
	return ABW_OK;
}
