// Context, error text and raw device-memory helpers of the C ABI.
#include "common.cuh"
#include <mutex>
#include <set>
#include <algorithm>
#include <cstring>

thread_local abw_ctx* abw_tls_ctx = nullptr;

namespace {
std::mutex g_live_mutex;
std::set<abw_ctx*> g_live;                                 // contexts that still exist: a buffer may be released after its context is gone
}

// ABW_REDZONE=1 (debug; the pool this was developed on refuses compute-sanitizer): every device block gets a 4 KiB canary zone on either side, is
// filled with 0xFF when handed out (a kernel that relies on memory it never wrote reads NaN / huge integers, and the bit-exact parity tests fail) and
// with 0xDD when released (use after free), is never reused, and the canaries are verified when the block is released or its context is destroyed.
// abw_redzone_violations() is the number of damaged canary zones seen so far in this process; ABW_REDZONE=abort also aborts at the first one.
namespace {
const size_t RZ = 4096;
struct RzBlock { unsigned char* base; size_t bytes; abw_ctx* ctx; };
std::map<void*, RzBlock> g_rz;
uint64_t g_rz_violations = 0;
int redzone_mode()
{
	static const int m = [] { const char* e = getenv("ABW_REDZONE"); return !e || !*e || strcmp(e, "0") == 0? 0 : strcmp(e, "abort") == 0? 2 : 1; }();
	return m;
}
}

__global__ void k_redzone_check(const unsigned char* __restrict__ front, const unsigned char* __restrict__ back, size_t nback, unsigned long long* bad)
{
	abw_grid_wait();
	// bad[0], bad[1]: damaged bytes before / after the block; bad[2], bad[3]: offset of the first one (atomicMin)
	for(size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < RZ + nback; i += (size_t)gridDim.x * blockDim.x) {
		const bool is_front = i < RZ;
		const size_t o = is_front? i : i - RZ;
		if((is_front? front[o] : back[o]) != 0xA5) {
			atomicAdd(&bad[is_front? 0 : 1], 1ull);
			atomicMin(&bad[is_front? 2 : 3], (unsigned long long)o);
		}
	}
}

static cudaError_t redzone_alloc(abw_ctx* ctx, size_t bytes, void** out)
{
	// the payload ends where the caller's size ends (rounded to 16 bytes only), so that one element past the end already lands on a canary
	const size_t payload = (bytes + 15) & ~(size_t)15;
	unsigned char* base = nullptr;
	cudaError_t e = cudaMallocAsync((void**)&base, RZ + payload + RZ, ctx->stream);
	if(e != cudaSuccess)
		return e;
	cudaMemsetAsync(base, 0xA5, RZ, ctx->stream);
	cudaMemsetAsync(base + RZ, 0xFF, payload, ctx->stream);
	cudaMemsetAsync(base + RZ + payload, 0xA5, RZ, ctx->stream);
	*out = base + RZ;
	std::lock_guard<std::mutex> lk(g_live_mutex);
	g_rz[*out] = RzBlock{base, payload, ctx};
	ctx->arena_misses++;
	return cudaGetLastError();
}

// verifies and releases one block (stream: the owning context's if it is still alive, else the default stream)
static void redzone_release(void* p, const RzBlock& b, cudaStream_t stream)
{
	unsigned long long* d_bad = nullptr;
	unsigned long long h_bad[4] = {0, 0, ~0ull, ~0ull};
	if(cudaMalloc((void**)&d_bad, sizeof(h_bad)) == cudaSuccess) {
		cudaMemcpyAsync(d_bad, h_bad, sizeof(h_bad), cudaMemcpyHostToDevice, stream);
		k_redzone_check<<<8, 256, 0, stream>>>(b.base, b.base + RZ + b.bytes, RZ, d_bad);
		cudaMemcpyAsync(h_bad, d_bad, sizeof(h_bad), cudaMemcpyDeviceToHost, stream);
		cudaMemsetAsync(b.base + RZ, 0xDD, b.bytes, stream);
		cudaStreamSynchronize(stream);
		cudaFree(d_bad);
	}
	if(h_bad[0] || h_bad[1]) {
		g_rz_violations++;
		fprintf(stderr, "ABW_REDZONE: block %p of %zu bytes: %llu byte(s) written before it (first at -%llu), %llu after it (first at +%llu)\n", p, b.bytes,
		        h_bad[0], h_bad[0]? (unsigned long long)RZ - h_bad[2] : 0ull, h_bad[1], h_bad[1]? (unsigned long long)b.bytes + h_bad[3] : 0ull);
		if(redzone_mode() == 2)
			abort();
	}
	cudaFreeAsync(b.base, stream);
}

cudaError_t abw_arena_alloc(abw_ctx* ctx, size_t bytes, void** out)
{
	if(!ctx)
		return cudaMalloc(out, bytes);
	if(redzone_mode())
		return redzone_alloc(ctx, bytes, out);
	// best fit among the cached blocks, as long as it does not waste more than a quarter of the block
	auto it = ctx->free_blocks.lower_bound(bytes);
	if(it != ctx->free_blocks.end() && it->first <= bytes + bytes / 4 + 65536) {
		*out = it->second;
		ctx->free_blocks.erase(it);
		return cudaSuccess;
	}
	// round up so that slightly different sizes of later passes (pair counts, cluster counts) still fit the cached block
	size_t cap = bytes;
	if(cap < 4096)
		cap = 4096;
	size_t step = 256;
	while(step * 16 < cap)
		step <<= 1;
	cap = (cap + step - 1) / step * step;
	ctx->arena_misses++;
	cudaError_t e = cudaMallocAsync(out, cap, ctx->stream);
	if(e != cudaSuccess) {
		// out of memory: give the cached blocks back and try once more
		cudaGetLastError();
		for(auto& kv : ctx->free_blocks) {
			cudaFreeAsync(kv.second, ctx->stream);
			ctx->block_cap.erase(kv.second);
		}
		ctx->free_blocks.clear();
		cudaStreamSynchronize(ctx->stream);
		e = cudaMallocAsync(out, cap, ctx->stream);
		if(e != cudaSuccess)
			return e;
	}
	ctx->block_cap[*out] = cap;
	return cudaSuccess;
}

// bytes from src to dst, one of them mapped pinned host memory; word-wise when both are 4-byte aligned
__global__ void k_copy_small(unsigned char* __restrict__ dst, const unsigned char* __restrict__ src, size_t bytes)
{
	abw_grid_wait();
	const size_t i0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x, stride = (size_t)gridDim.x * blockDim.x;
	if(((reinterpret_cast<uintptr_t>(dst) | reinterpret_cast<uintptr_t>(src)) & 3u) == 0) {
		const size_t words = bytes >> 2;
		for(size_t i = i0; i < words; i += stride)
			reinterpret_cast<uint32_t*>(dst)[i] = reinterpret_cast<const uint32_t*>(src)[i];
		for(size_t i = (words << 2) + i0; i < bytes; i += stride)
			dst[i] = src[i];
	}
	else {
		for(size_t i = i0; i < bytes; i += stride)
			dst[i] = src[i];
	}
}

static cudaError_t copy_small(abw_ctx* ctx, void* dst, const void* src, size_t bytes)
{
	const unsigned int blocks = (unsigned int)std::min<size_t>(64, (bytes / 4 + 255) / 256 + 1);
	abw_launch_pdl(k_copy_small, blocks, 256, 0, ctx->stream, (unsigned char*)dst, (const unsigned char*)src, bytes);      // in the middle of the chain of ABW_LAUNCH kernels
	ctx->launches++;
	return cudaGetLastError();
}

cudaError_t abw_fetch(abw_ctx* ctx, void* h_dst, const void* d_src, size_t bytes)
{
	if(bytes == 0)
		return cudaSuccess;
	if(bytes <= ((size_t)256 << 10)) {
		if(!ctx->h_bounce) {
			ctx->bounce_cap = (size_t)2 << 20;
			if(cudaHostAlloc((void**)&ctx->h_bounce, ctx->bounce_cap, cudaHostAllocMapped) != cudaSuccess) {
				cudaGetLastError();
				ctx->h_bounce = nullptr;
				ctx->bounce_cap = 0;
			}
		}
		const size_t need = (bytes + 255) & ~(size_t)255;
		if(ctx->h_bounce && ctx->bounce_used + need <= ctx->bounce_cap) {
			unsigned char* slot = ctx->h_bounce + ctx->bounce_used;
			ctx->bounce_used += need;
			ctx->pending.push_back({h_dst, slot, bytes});
			return copy_small(ctx, slot, d_src, bytes);
		}
	}
	return cudaMemcpyAsync(h_dst, d_src, bytes, cudaMemcpyDeviceToHost, ctx->stream);
}

cudaError_t abw_sync(abw_ctx* ctx)
{
	cudaError_t e = cudaStreamSynchronize(ctx->stream);
	if(e == cudaSuccess && *ctx->scan_failed) {
		*ctx->scan_failed = 0;
		e = cudaErrorTimeout;
	}
	if(e == cudaSuccess)
		for(const abw_ctx::Fetch& f : ctx->pending)
			memcpy(f.h_dst, f.slot, f.bytes);
	ctx->pending.clear();
	ctx->bounce_used = 0;
	ctx->stage_used = 0;
	return e;
}

cudaError_t abw_upload_small(abw_ctx* ctx, void* d_dst, const void* h_src, size_t bytes)
{
	if(bytes == 0)
		return cudaSuccess;
	if(!ctx->h_stage) {
		ctx->stage_cap = (size_t)4 << 20;
		if(cudaMallocHost((void**)&ctx->h_stage, ctx->stage_cap) != cudaSuccess) {
			cudaGetLastError();
			ctx->h_stage = nullptr;
			ctx->stage_cap = 0;
		}
	}
	const size_t need = (bytes + 255) & ~(size_t)255;
	if(ctx->h_stage && ctx->stage_used + need <= ctx->stage_cap) {
		unsigned char* slot = ctx->h_stage + ctx->stage_used;
		memcpy(slot, h_src, bytes);
		ctx->stage_used += need;
		return copy_small(ctx, d_dst, slot, bytes);            // pinned memory is mapped into the device's address space (unified addressing)
	}
	return cudaMemcpyAsync(d_dst, h_src, bytes, cudaMemcpyHostToDevice, ctx->stream);      // does not fit the staging area: the driver stages it
}

void abw_arena_free(abw_ctx* ctx, void* p)
{
	if(!p)
		return;
	bool alive = false;
	RzBlock rz{nullptr, 0, nullptr};
	{
		std::lock_guard<std::mutex> lk(g_live_mutex);
		alive = ctx && g_live.count(ctx) != 0;
		auto it = g_rz.find(p);
		if(it != g_rz.end()) {
			rz = it->second;
			g_rz.erase(it);
		}
	}
	if(rz.base) {
		redzone_release(p, rz, alive? ctx->stream : (cudaStream_t)0);
		return;
	}
	if(!alive) {
		cudaFree(p);
		return;
	}
	auto it = ctx->block_cap.find(p);
	if(it == ctx->block_cap.end()) {
		cudaFreeAsync(p, ctx->stream);
		return;
	}
	ctx->free_blocks.insert(std::make_pair(it->second, p));
}

extern "C" {

const char* abw_version(void) { return "abawaca_b200 0.2 (sm_100a)"; }

void abw_default_params(abw_params* p)
{
	if(!p)
		return;
	p->cluster_ndps_threshold = 100;
	p->sensitivity_threshold = 0.8;
	p->specificity_threshold = 0.8;
	p->product_threshold = 0.8;
	p->sum_threshold = 1.6;
	p->scg_overlap_threshold = 0.2;
	p->scg_min_size = 500000;
	p->fraction_dps_in = 0.8;
	p->split_scaf_ratio_threshold = 0.1;
	p->max_snps = 15;
	p->window_size = 2000;
	p->min_reported_score = 0.8;
}

int abw_ctx_create(int device, abw_ctx** out)
{
	if(!out)
		return ABW_ERR_ARG;
	*out = nullptr;
	int ndev = 0;
	if(cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
		return ABW_ERR_CUDA;        // no CPU fallback: without a device there is no context
	if(device < 0 || device >= ndev)
		return ABW_ERR_ARG;
	if(cudaSetDevice(device) != cudaSuccess)
		return ABW_ERR_CUDA;
	abw_ctx* c = new abw_ctx();
	c->device = device;
	if(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) != cudaSuccess ||
	   cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking) != cudaSuccess ||
	   cudaHostAlloc((void**)&c->scan_failed, sizeof(uint32_t), cudaHostAllocMapped) != cudaSuccess) {
		delete c;
		return ABW_ERR_CUDA;
	}
	*c->scan_failed = 0;
	cudaDeviceProp prop;
	if(cudaGetDeviceProperties(&prop, device) == cudaSuccess)
		c->sm_count = prop.multiProcessorCount;
	// keep freed blocks in the pool instead of returning them to the driver at every synchronisation
	cudaMemPool_t pool;
	if(cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
		uint64_t keep = UINT64_MAX;
		cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
	}
	{
		std::lock_guard<std::mutex> lk(g_live_mutex);
		g_live.insert(c);
	}
	*out = c;
	return ABW_OK;
}

void abw_ctx_destroy(abw_ctx* ctx)
{
	if(!ctx)
		return;
	cudaSetDevice(ctx->device);
	{
		std::lock_guard<std::mutex> lk(g_live_mutex);
		g_live.erase(ctx);
	}
	cudaStreamSynchronize(ctx->stream);
	if(redzone_mode()) {
		// blocks this context handed out that are still held (search handles released later, leaks): verify their canaries now, while the stream exists
		std::vector<std::pair<void*, RzBlock>> mine;
		{
			std::lock_guard<std::mutex> lk(g_live_mutex);
			for(auto& kv : g_rz)
				if(kv.second.ctx == ctx)
					mine.push_back(kv);
		}
		for(auto& kv : mine) {
			RzBlock keep = kv.second;
			unsigned long long* d_bad = nullptr;
			unsigned long long h_bad[4] = {0, 0, ~0ull, ~0ull};
			if(cudaMalloc((void**)&d_bad, sizeof(h_bad)) == cudaSuccess) {
				cudaMemcpy(d_bad, h_bad, sizeof(h_bad), cudaMemcpyHostToDevice);
				k_redzone_check<<<8, 256, 0, ctx->stream>>>(keep.base, keep.base + RZ + keep.bytes, RZ, d_bad);
				cudaStreamSynchronize(ctx->stream);
				cudaMemcpy(h_bad, d_bad, sizeof(h_bad), cudaMemcpyDeviceToHost);
				cudaFree(d_bad);
			}
			if(h_bad[0] || h_bad[1]) {
				g_rz_violations++;
				fprintf(stderr, "ABW_REDZONE: live block %p of %zu bytes damaged at context destruction (%llu before, %llu after)\n", kv.first, keep.bytes, h_bad[0], h_bad[1]);
				if(redzone_mode() == 2)
					abort();
			}
			std::lock_guard<std::mutex> lk(g_live_mutex);
			auto it = g_rz.find(kv.first);
			if(it != g_rz.end())
				it->second.ctx = nullptr;
		}
	}
	for(auto& kv : ctx->free_blocks)
		cudaFree(kv.second);
	ctx->free_blocks.clear();
	if(ctx->h_stage)
		cudaFreeHost(ctx->h_stage);
	ctx->h_stage = nullptr;
	if(ctx->h_bounce)
		cudaFreeHost(ctx->h_bounce);
	ctx->h_bounce = nullptr;
	if(ctx->h_prog)
		cudaFreeHost(ctx->h_prog);
	ctx->h_prog = nullptr;
	if(ctx->scan_scratch)
		cudaFree(ctx->scan_scratch);
	ctx->scan_scratch = nullptr;
	if(ctx->scan_failed)
		cudaFreeHost(ctx->scan_failed);
	ctx->scan_failed = nullptr;
	for(cudaEvent_t e : ctx->copy_events)
		cudaEventDestroy(e);
	if(ctx->side_stream) {
		cudaStreamSynchronize(ctx->side_stream);
		cudaStreamDestroy(ctx->side_stream);
		cudaEventDestroy(ctx->ev_fork);
		cudaEventDestroy(ctx->ev_join);
	}
	if(ctx->copy_stream)
		cudaStreamDestroy(ctx->copy_stream);
	if(ctx->stream)
		cudaStreamDestroy(ctx->stream);
	if(ctx->ev_a) {
		cudaEventDestroy(ctx->ev_a);
		cudaEventDestroy(ctx->ev_b);
	}
	delete ctx;
}

const char* abw_last_error(const abw_ctx* ctx) { return ctx? ctx->err.c_str() : "no context (is a CUDA device present?)"; }

uint64_t abw_kernel_launches(const abw_ctx* ctx) { return ctx? ctx->launches : 0; }

uint64_t abw_arena_misses(const abw_ctx* ctx) { return ctx? ctx->arena_misses : 0; }

uint64_t abw_redzone_violations(void) { return g_rz_violations; }

void* abw_ctx_stream(const abw_ctx* ctx) { return ctx? (void*)ctx->stream : nullptr; }

int abw_ctx_synchronize(abw_ctx* ctx)
{
	if(!ctx)
		return ABW_ERR_ARG;
	ABW_CUDA(ctx, cudaStreamSynchronize(ctx->copy_stream));
	ABW_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
	for(cudaEvent_t e : ctx->copy_events)      // every staged copy has completed: tickets handed out so far are retired
		cudaEventDestroy(e);
	ctx->copy_retired += ctx->copy_events.size();      // tickets stay monotonic: a retired one is simply "already complete"
	ctx->copy_events.clear();
	return ABW_OK;
}

int abw_profile_enable(abw_ctx* ctx, int on)
{
	if(!ctx)
		return ABW_ERR_ARG;
	if(on && !ctx->ev_a) {
		ABW_CUDA(ctx, cudaEventCreate(&ctx->ev_a));
		ABW_CUDA(ctx, cudaEventCreate(&ctx->ev_b));
	}
	ctx->profiling = on != 0;
	if(on)
		ctx->prof.clear();
	return ABW_OK;
}

size_t abw_profile_report(abw_ctx* ctx, char* buf, size_t cap)
{
	if(!ctx)
		return 0;
	std::string out;
	char line[256];
	for(auto& kv : ctx->prof) {
		snprintf(line, sizeof(line), "%s\t%llu\t%.6f\n", kv.first.c_str(), (unsigned long long)kv.second.first, kv.second.second);
		out += line;
	}
	if(buf && cap) {
		size_t n = std::min(out.size(), cap - 1);
		memcpy(buf, out.data(), n);
		buf[n] = 0;
	}
	return out.size() + 1;
}

int abw_device_alloc(abw_ctx* ctx, size_t bytes, void** d_out)
{
	if(!ctx || !d_out)
		return abw_fail(ctx, ABW_ERR_ARG, "abw_device_alloc: null argument");
	ABW_ENTER(ctx);
	ABW_CUDA(ctx, abw_arena_alloc(ctx, bytes? bytes : 1, d_out));
	ABW_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
	return ABW_OK;
}

int abw_device_free(abw_ctx* ctx, void* d_ptr)
{
	if(!ctx)
		return ABW_ERR_ARG;
	abw_arena_free(ctx, d_ptr);                            // cached for reuse in the order of the context stream
	return ABW_OK;
}

int abw_copy_to_device(abw_ctx* ctx, void* d_dst, const void* h_src, size_t bytes)
{
	if(!ctx)
		return ABW_ERR_ARG;
	ABW_CUDA(ctx, cudaMemcpyAsync(d_dst, h_src, bytes, cudaMemcpyHostToDevice, ctx->stream));
	ABW_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
	return ABW_OK;
}

int abw_copy_to_host(abw_ctx* ctx, void* h_dst, const void* d_src, size_t bytes)
{
	if(!ctx)
		return ABW_ERR_ARG;
	ABW_CUDA(ctx, cudaMemcpyAsync(h_dst, d_src, bytes, cudaMemcpyDeviceToHost, ctx->stream));
	ABW_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
	return ABW_OK;
}

int abw_h2d_async(abw_ctx* ctx, void* d_dst, const void* h_src, size_t bytes, uint64_t* ticket)
{
	if(!ctx || !ticket)
		return abw_fail(ctx, ABW_ERR_ARG, "abw_h2d_async: null argument");
	// the destination may have been allocated in order on the compute stream: let the copy stream see that allocation
	cudaEvent_t ready;
	ABW_CUDA(ctx, cudaEventCreateWithFlags(&ready, cudaEventDisableTiming));
	ABW_CUDA(ctx, cudaEventRecord(ready, ctx->stream));
	ABW_CUDA(ctx, cudaStreamWaitEvent(ctx->copy_stream, ready, 0));
	ABW_CUDA(ctx, cudaEventDestroy(ready));
	ABW_CUDA(ctx, cudaMemcpyAsync(d_dst, h_src, bytes, cudaMemcpyHostToDevice, ctx->copy_stream));
	cudaEvent_t done;
	ABW_CUDA(ctx, cudaEventCreateWithFlags(&done, cudaEventDisableTiming));
	ABW_CUDA(ctx, cudaEventRecord(done, ctx->copy_stream));
	ctx->copy_events.push_back(done);
	*ticket = ctx->copy_retired + ctx->copy_events.size();      // 1-based and monotonic over the life of the context; 0 means "nothing to wait for"
	return ABW_OK;
}

int abw_d2h_async(abw_ctx* ctx, void* h_dst, const void* d_src, size_t bytes)
{
	if(!ctx || (!h_dst && bytes) || (!d_src && bytes))
		return abw_fail(ctx, ABW_ERR_ARG, "abw_d2h_async: null argument");
	// everything enqueued on the compute stream so far produces d_src; later compute overlaps the copy
	cudaEvent_t ready;
	ABW_CUDA(ctx, cudaEventCreateWithFlags(&ready, cudaEventDisableTiming));
	ABW_CUDA(ctx, cudaEventRecord(ready, ctx->stream));
	ABW_CUDA(ctx, cudaStreamWaitEvent(ctx->copy_stream, ready, 0));
	ABW_CUDA(ctx, cudaEventDestroy(ready));
	ABW_CUDA(ctx, cudaMemcpyAsync(h_dst, d_src, bytes, cudaMemcpyDeviceToHost, ctx->copy_stream));
	return ABW_OK;
}

int abw_wait_h2d(abw_ctx* ctx, uint64_t ticket)
{
	if(!ctx || ticket > ctx->copy_retired + ctx->copy_events.size())
		return abw_fail(ctx, ABW_ERR_ARG, "abw_wait_h2d: unknown ticket");
	if(ticket <= ctx->copy_retired)                    // 0, or retired by an abw_ctx_synchronize since it was issued: the copy has completed
		return ABW_OK;
	ABW_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, ctx->copy_events[ticket - ctx->copy_retired - 1], 0));
	return ABW_OK;
}

int abw_memset_device(abw_ctx* ctx, void* d_ptr, int byte, size_t bytes)
{
	if(!ctx)
		return ABW_ERR_ARG;
	ABW_CUDA(ctx, cudaMemsetAsync(d_ptr, byte, bytes, ctx->stream));
	return ABW_OK;
}

}  // extern "C"
