// Device-wide exclusive scan and a stable LSD radix sort (8-bit digits), hand-written for sm_100a.
//
// The sort is used once per split-search problem (every Dimension is sorted once, not once per
// cluster as std::sort in ClusterSeparatorBySensitivitySpecificity.cpp:114 does) and once per sample in
// the coverage stage (reads grouped by segment while keeping SAM order).  Stability matters for the
// latter: coverage is an order-dependent fp64 sum (SURVEY.md quirk Q5).
#include "common.cuh"

namespace {

constexpr int SCAN_THREADS = 256;
constexpr int SCAN_ITEMS = 8;
constexpr int SCAN_TILE = SCAN_THREADS * SCAN_ITEMS;

__device__ __forceinline__ uint64_t warp_incl_scan_u64(uint64_t v)
{
	int lane = threadIdx.x & 31;
#pragma unroll
	for(int o = 1; o < 32; o <<= 1) {
		uint64_t t = __shfl_up_sync(0xffffffffu, v, o);
		if(lane >= o)
			v += t;
	}
	return v;
}

// block-wide exclusive scan of one value per thread; returns exclusive prefix, *total = block sum
__device__ __forceinline__ uint64_t block_excl_scan_u64(uint64_t v, uint64_t* total, uint64_t* smem /* [33] */)
{
	int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
	uint64_t incl = warp_incl_scan_u64(v);
	if(lane == 31)
		smem[warp] = incl;
	__syncthreads();
	if(warp == 0) {
		uint64_t w = (lane < nw)? smem[lane] : 0;
		uint64_t wi = warp_incl_scan_u64(w);
		smem[lane] = wi - w;
		if(lane == 31)
			smem[32] = wi;
	}
	__syncthreads();
	uint64_t r = smem[warp] + incl - v;
	*total = smem[32];
	__syncthreads();
	return r;
}

// One pass, one launch: tiles of SCAN_TILE values are handed out by ticket (a tile only ever waits for tiles drawn earlier by CTAs that are running);
// a tile publishes its sum, looks back over its predecessors until it meets a published inclusive prefix, publishes its own and writes its values.
// The per-context scratch (status words, sums, prefixes, ticket) is never cleared between scans: status words carry the number of the scan that wrote
// them (epoch), and the ticket counter keeps running -- the host knows how many tickets every scan draws (its number of CTAs = tiles).
// A look-back wait that gives up sets *failed (mapped pinned memory of the context), which abw_sync reports.
template <typename Tin>
__global__ void __launch_bounds__(SCAN_THREADS) k_scan_onepass(const Tin* __restrict__ in, uint64_t* __restrict__ out, uint64_t n, uint64_t* __restrict__ total_out,
                                                              unsigned long long* __restrict__ ticket, unsigned long long ticket_base, uint32_t epoch,
                                                              uint32_t* __restrict__ status, unsigned long long* __restrict__ aggs, unsigned long long* __restrict__ prefixes,
                                                              uint32_t* __restrict__ failed)
{
	abw_grid_wait();
	__shared__ uint64_t sm[33];
	__shared__ unsigned long long sm_tile, sm_carry;
	if(threadIdx.x == 0)
		sm_tile = atomicAdd(ticket, 1ull) - ticket_base;
	__syncthreads();
	abw_launch_dependents();                               // tile drawn: once every CTA has one, the next kernel may take the slots they free
	const uint64_t tile = sm_tile;
	const uint64_t base = tile * SCAN_TILE + (uint64_t)threadIdx.x * SCAN_ITEMS;
	uint64_t v[SCAN_ITEMS];
	uint64_t s = 0;
#pragma unroll
	for(int i = 0; i < SCAN_ITEMS; i++) {
		v[i] = (base + i < n)? (uint64_t)in[base + i] : 0;
		s += v[i];
	}
	uint64_t total;
	uint64_t ex = block_excl_scan_u64(s, &total, sm);
	if(threadIdx.x < 32) {
		const int lane = threadIdx.x;
		unsigned long long carry = 0;
		if(tile > 0) {
			if(lane == 0) {
				__stcg(&aggs[tile], (unsigned long long)total);
				lb_split_publish(&status[tile], LB_AGG, epoch);
			}
			const bool ok = lb_walk(tile, (uint32_t)tile, [&](uint64_t i) { return ld_volatile_u32(&status[i]); }, [&](uint32_t raw) { return lb_split_state(raw, epoch); },
			                        [&](uint32_t, uint64_t i, bool take, uint32_t first_prefix) {
				unsigned long long x = lb_split_value<unsigned long long>(i, take, (uint32_t)lane == first_prefix, aggs, prefixes,
				                                                          [](const unsigned long long* p) { return __ldcg(p); });
#pragma unroll
				for(int o = 16; o > 0; o >>= 1)
					x += __shfl_xor_sync(0xffffffffu, x, o);
				carry += x;
			});
			if(!ok && lane == 0)
				*failed = 1u;
		}
		if(lane == 0) {
			__stcg(&prefixes[tile], carry + (unsigned long long)total);
			lb_split_publish(&status[tile], LB_PREFIX, epoch);
			sm_carry = carry;
			if(total_out != nullptr && tile == gridDim.x - 1)
				*total_out = carry + total;
		}
	}
	__syncthreads();
	ex += sm_carry;
#pragma unroll
	for(int i = 0; i < SCAN_ITEMS; i++) {
		if(base + i < n)
			out[base + i] = ex;
		ex += v[i];
	}
}

template <typename Tin>
int scan_impl(abw_ctx* ctx, const Tin* d_in, uint64_t* d_out, uint64_t n, uint64_t* d_total)
{
	if(n == 0) {
		if(d_total)
			ABW_CUDA(ctx, cudaMemsetAsync(d_total, 0, sizeof(uint64_t), ctx->stream));
		return ABW_OK;
	}
	const unsigned int nblocks = abw_div_up(n, SCAN_TILE);
	// scratch of the context, grown on demand (scans of one context run one after the other on its stream)
	if(ctx->scan_cap < nblocks) {
		size_t cap = 4096;
		while(cap < nblocks)
			cap <<= 1;
		if(ctx->scan_scratch)
			ABW_CUDA(ctx, cudaFreeAsync(ctx->scan_scratch, ctx->stream));
		ABW_CUDA(ctx, cudaMallocAsync(&ctx->scan_scratch, cap * 20 + 64, ctx->stream));
		ABW_CUDA(ctx, cudaMemsetAsync(ctx->scan_scratch, 0, cap * 20 + 64, ctx->stream));
		ctx->scan_cap = cap;
		ctx->scan_epoch = 0;
		ctx->scan_tickets = 0;
	}
	unsigned char* base = (unsigned char*)ctx->scan_scratch;
	unsigned long long* ticket = (unsigned long long*)base;
	unsigned long long* aggs = (unsigned long long*)(base + 64);
	unsigned long long* prefixes = aggs + ctx->scan_cap;
	uint32_t* status = (uint32_t*)(prefixes + ctx->scan_cap);
	ctx->scan_epoch++;
	if(ctx->scan_epoch >= (1u << 30)) {                    // the epoch field of the status words would wrap: start over
		ABW_CUDA(ctx, cudaMemsetAsync(ctx->scan_scratch, 0, ctx->scan_cap * 20 + 64, ctx->stream));
		ctx->scan_epoch = 1;
		ctx->scan_tickets = 0;
	}
	ABW_LAUNCH(ctx, k_scan_onepass<Tin>, nblocks, SCAN_THREADS, 0, d_in, d_out, n, d_total, ticket, (unsigned long long)ctx->scan_tickets, ctx->scan_epoch, status, aggs,
	           prefixes, ctx->scan_failed);
	ctx->scan_tickets += nblocks;
	return ABW_OK;
}

// ---------------------------------------------------------------------------------------------------
// radix sort
// ---------------------------------------------------------------------------------------------------
constexpr int RS_THREADS = 256;
constexpr int RS_WARPS = RS_THREADS / 32;
constexpr int RS_ITEMS = 8;                        // keys per lane
constexpr int RS_WARP_TILE = 32 * RS_ITEMS;        // 512
constexpr int RS_TILE = RS_THREADS * RS_ITEMS;     // 4096

template <typename K>
__global__ void __launch_bounds__(RS_THREADS) k_rs_or_and(const K* __restrict__ keys, uint64_t n, uint64_t stride, unsigned long long* __restrict__ or_and)
{
	abw_grid_wait();
	const K* a = keys + (uint64_t)blockIdx.y * stride;
	unsigned long long o = 0, an = ~0ull;
	for(uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
		unsigned long long k = (unsigned long long)a[i];
		o |= k;
		an &= k;
	}
#pragma unroll
	for(int s = 16; s > 0; s >>= 1) {
		o |= __shfl_xor_sync(0xffffffffu, o, s);
		an &= __shfl_xor_sync(0xffffffffu, an, s);
	}
	if((threadIdx.x & 31) == 0) {
		atomicOr(&or_and[0], o);
		atomicAnd(&or_and[1], an);
	}
}

// per-block digit histogram, layout hist[((array * NB) + digit) * nblocks + block], NB = 2^BITS digits
template <typename K, int BITS>
__global__ void __launch_bounds__(RS_THREADS) k_rs_hist(const K* __restrict__ keys, uint64_t n, uint64_t stride, int shift, uint32_t* __restrict__ hist)
{
	abw_grid_wait();
	constexpr int NB = 1 << BITS;
	__shared__ uint32_t sh[NB];
	const K* a = keys + (uint64_t)blockIdx.y * stride;
	for(int d = threadIdx.x; d < NB; d += RS_THREADS)
		sh[d] = 0;
	__syncthreads();
	uint64_t base = (uint64_t)blockIdx.x * RS_TILE;
#pragma unroll
	for(int r = 0; r < RS_ITEMS; r++) {
		uint64_t i = base + (uint64_t)r * RS_THREADS + threadIdx.x;
		if(i < n)
			atomicAdd(&sh[(uint32_t)(a[i] >> shift) & (uint32_t)(NB - 1)], 1u);
	}
	__syncthreads();
	for(int d = threadIdx.x; d < NB; d += RS_THREADS)
		hist[((uint64_t)blockIdx.y * NB + d) * gridDim.x + blockIdx.x] = sh[d];
}

template <typename K, int BITS>
__global__ void __launch_bounds__(RS_THREADS) k_rs_scatter(const K* __restrict__ keys_in, const uint32_t* __restrict__ vals_in, K* __restrict__ keys_out,
                                                          uint32_t* __restrict__ vals_out, uint64_t n, uint64_t stride, int shift, const uint64_t* __restrict__ offsets)
{
	abw_grid_wait();
	constexpr int NB = 1 << BITS;
	__shared__ uint32_t cnt[RS_WARPS][NB + 1];
	__shared__ uint64_t digit_base[NB];
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	const uint64_t arr = blockIdx.y;
	const K* ki = keys_in + arr * stride;
	const uint32_t* vi = vals_in + arr * stride;
	K* ko = keys_out + arr * stride;
	uint32_t* vo = vals_out + arr * stride;
	for(int d = lane; d < NB + 1; d += 32)
		cnt[warp][d] = 0;
	__syncwarp();
	K key[RS_ITEMS];
	uint32_t val[RS_ITEMS];
	uint32_t lrank[RS_ITEMS];
	const uint64_t wbase = (uint64_t)blockIdx.x * RS_TILE + (uint64_t)warp * RS_WARP_TILE;
	const uint32_t lt = (1u << lane) - 1u;
#pragma unroll
	for(int r = 0; r < RS_ITEMS; r++) {
		uint64_t i = wbase + (uint64_t)r * 32 + lane;
		bool ok = i < n;
		key[r] = ok? ki[i] : (K)0;
		val[r] = ok? vi[i] : 0u;
	}
	// phase A: stable rank of every key among the keys of its warp with the same digit
#pragma unroll
	for(int r = 0; r < RS_ITEMS; r++) {
		uint64_t i = wbase + (uint64_t)r * 32 + lane;
		uint32_t d = (i < n)? ((uint32_t)(key[r] >> shift) & (uint32_t)(NB - 1)) : (uint32_t)NB;
		uint32_t peers = __match_any_sync(0xffffffffu, d);
		int leader = __ffs(peers) - 1;
		uint32_t old = 0;
		if(lane == leader) {
			old = cnt[warp][d];
			cnt[warp][d] = old + __popc(peers);
		}
		old = __shfl_sync(0xffffffffu, old, leader);
		lrank[r] = old + __popc(peers & lt);
		__syncwarp();
	}
	__syncthreads();
	// phase B: every digit gets the destination base of each (warp, digit)
	for(int d = threadIdx.x; d < NB; d += RS_THREADS) {
		digit_base[d] = offsets[(arr * NB + d) * gridDim.x + blockIdx.x] - arr * n;
		uint32_t acc = 0;
#pragma unroll
		for(int w = 0; w < RS_WARPS; w++) {
			uint32_t c = cnt[w][d];
			cnt[w][d] = acc;
			acc += c;
		}
	}
	__syncthreads();
	// phase C
#pragma unroll
	for(int r = 0; r < RS_ITEMS; r++) {
		uint64_t i = wbase + (uint64_t)r * 32 + lane;
		if(i < n) {
			uint32_t dg = (uint32_t)(key[r] >> shift) & (uint32_t)(NB - 1);
			uint64_t dst = digit_base[dg] + cnt[warp][dg] + lrank[r];
			ko[dst] = key[r];
			vo[dst] = val[r];
		}
	}
}

template <typename K, int BITS>
int radix_pass(abw_ctx* ctx, const K* src_k, const uint32_t* src_v, K* dst_k, uint32_t* dst_v, uint64_t n, uint32_t batch, uint64_t stride, int shift,
               unsigned int nblocks, uint32_t* hist, uint64_t* offs)
{
	dim3 grid(nblocks, batch);
	const uint64_t nh = (uint64_t)batch * (1u << BITS) * nblocks;
	ABW_LAUNCH(ctx, (k_rs_hist<K, BITS>), grid, RS_THREADS, 0, src_k, n, stride, shift, hist);
	ABW_CHECK(abw_exclusive_scan_u32_to_u64(ctx, hist, offs, nh, nullptr));
	ABW_LAUNCH(ctx, (k_rs_scatter<K, BITS>), grid, RS_THREADS, 0, src_k, src_v, dst_k, dst_v, n, stride, shift, offs);
	return ABW_OK;
}

template <typename K>
int radix_sort_impl(abw_ctx* ctx, K* d_keys, K* d_keys_tmp, uint32_t* d_vals, uint32_t* d_vals_tmp, uint64_t n, uint32_t batch, uint64_t stride, int nbits,
                    const unsigned long long* known_varying = nullptr)
{
	if(n == 0 || batch == 0 || nbits == 0)
		return ABW_OK;
	unsigned int nblocks = abw_div_up(n, RS_TILE);
	unsigned long long varying;
	if(known_varying) {
		// the caller looked at the keys while it made them
		varying = *known_varying;
		if(nbits > 0 && nbits < 64)
			varying &= (1ull << nbits) - 1ull;
		if(varying == 0)
			return ABW_OK;                                  // all keys equal: already sorted (stable)
	}
	else if(nbits < 0) {
		// the caller knows that every key bit below -nbits varies (dense ids): no inspection pass, no host round trip
		nbits = -nbits;
		varying = (nbits < 64)? ((1ull << nbits) - 1ull) : ~0ull;
	}
	else {
		DevBuf<unsigned long long> or_and;
		ABW_CUDA(ctx, or_and.alloc(2));
		unsigned long long init[2] = {0ull, ~0ull};
		ABW_CUDA(ctx, cudaMemcpyAsync(or_and.p, init, sizeof(init), cudaMemcpyHostToDevice, ctx->stream));
		{
			dim3 grid(min(nblocks, 4u * (unsigned)ctx->sm_count), batch);
			ABW_LAUNCH(ctx, k_rs_or_and<K>, grid, RS_THREADS, 0, d_keys, n, stride, or_and.p);
		}
		unsigned long long oa[2];
		ABW_CUDA(ctx, abw_fetch(ctx, oa, or_and.p, sizeof(oa)));
		ABW_CUDA(ctx, abw_sync(ctx));
		varying = oa[0] ^ oa[1];
		if(nbits < 64)
			varying &= (1ull << nbits) - 1ull;
	}
	// plan: cover every varying bit with as few 8- or 9-bit digits as possible (bits that are equal in all keys are skipped)
	struct Pass { int shift, bits; };
	Pass plan[16];
	int npass = 0;
	{
		int total[11] = {0};
		for(int width = 8; width <= 10; width++) {
			int cnt = 0, bit = 0;
			while(bit < 64) {
				if(!((varying >> bit) & 1ull)) { bit++; continue; }
				cnt++;
				bit += width;
			}
			total[width] = cnt;
		}
		// the narrowest digit that needs the fewest passes; 10-bit digits measured slower than two 8-bit passes (1024 bins: a third of the CTAs per SM in the
		// scatter and four times the histogram to scan), so they are only planned when they save two passes
		int width = 8;
		if(total[9] < total[width])
			width = 9;
		if(total[10] + 1 < total[width])
			width = 10;
		int bit = 0;
		while(bit < 64) {
			if(!((varying >> bit) & 1ull)) { bit++; continue; }
			plan[npass].shift = bit;
			plan[npass].bits = width;
			npass++;
			bit += width;
		}
	}
	DevBuf<uint32_t> hist;
	DevBuf<uint64_t> offs;
	uint64_t nh = (uint64_t)batch * 1024 * nblocks;
	ABW_CUDA(ctx, hist.alloc(nh));
	ABW_CUDA(ctx, offs.alloc(nh));
	K* src_k = d_keys; K* dst_k = d_keys_tmp;
	uint32_t* src_v = d_vals; uint32_t* dst_v = d_vals_tmp;
	for(int ps = 0; ps < npass; ps++) {
		if(plan[ps].bits == 10)
			ABW_CHECK((radix_pass<K, 10>(ctx, src_k, src_v, dst_k, dst_v, n, batch, stride, plan[ps].shift, nblocks, hist.p, offs.p)));
		else if(plan[ps].bits == 9)
			ABW_CHECK((radix_pass<K, 9>(ctx, src_k, src_v, dst_k, dst_v, n, batch, stride, plan[ps].shift, nblocks, hist.p, offs.p)));
		else
			ABW_CHECK((radix_pass<K, 8>(ctx, src_k, src_v, dst_k, dst_v, n, batch, stride, plan[ps].shift, nblocks, hist.p, offs.p)));
		K* tk = src_k; src_k = dst_k; dst_k = tk;
		uint32_t* tv = src_v; src_v = dst_v; dst_v = tv;
	}
	if(src_k != d_keys) {
		uint64_t total = (uint64_t)(batch - 1) * stride + n;
		ABW_CUDA(ctx, cudaMemcpyAsync(d_keys, src_k, total * sizeof(K), cudaMemcpyDeviceToDevice, ctx->stream));
		ABW_CUDA(ctx, cudaMemcpyAsync(d_vals, src_v, total * sizeof(uint32_t), cudaMemcpyDeviceToDevice, ctx->stream));
	}
	return ABW_OK;
}

}  // namespace

int abw_exclusive_scan_u64(abw_ctx* ctx, const uint64_t* d_in, uint64_t* d_out, uint64_t n, uint64_t* d_total)
{
	return scan_impl<uint64_t>(ctx, d_in, d_out, n, d_total);
}

int abw_exclusive_scan_u32_to_u64(abw_ctx* ctx, const uint32_t* d_in, uint64_t* d_out, uint64_t n, uint64_t* d_total)
{
	return scan_impl<uint32_t>(ctx, d_in, d_out, n, d_total);
}

int abw_radix_sort_pairs_u64(abw_ctx* ctx, uint64_t* d_keys, uint64_t* d_keys_tmp, uint32_t* d_vals, uint32_t* d_vals_tmp, uint64_t n, uint32_t batch,
                             uint64_t stride, int nbits)
{
	return radix_sort_impl<uint64_t>(ctx, d_keys, d_keys_tmp, d_vals, d_vals_tmp, n, batch, stride, nbits);
}

int abw_radix_sort_pairs_u32(abw_ctx* ctx, uint32_t* d_keys, uint32_t* d_keys_tmp, uint32_t* d_vals, uint32_t* d_vals_tmp, uint64_t n, uint32_t batch,
                             uint64_t stride, int nbits)
{
	return radix_sort_impl<uint32_t>(ctx, d_keys, d_keys_tmp, d_vals, d_vals_tmp, n, batch, stride, nbits);
}

int abw_radix_sort_pairs_u32_varying(abw_ctx* ctx, uint32_t* d_keys, uint32_t* d_keys_tmp, uint32_t* d_vals, uint32_t* d_vals_tmp, uint64_t n, uint32_t batch,
                                     uint64_t stride, unsigned long long varying)
{
	return radix_sort_impl<uint32_t>(ctx, d_keys, d_keys_tmp, d_vals, d_vals_tmp, n, batch, stride, 32, &varying);
}
