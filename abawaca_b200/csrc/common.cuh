// Shared host/device helpers of libabawaca_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <nvtx3/nvToolsExt.h>      // header only: ranges cost nothing unless a tool (nsys, ncu --nvtx) is attached
#include <stdint.h>
#include <string>
#include <vector>
#include <map>
#include <utility>
#include <cstdio>
#include "../../include/abawaca_b200.h"

struct abw_ctx {
	int          device = 0;
	cudaStream_t stream = nullptr;
	cudaStream_t copy_stream = nullptr;       // host->device staging that overlaps kernels of `stream` (abw_h2d_async)
	cudaStream_t side_stream = nullptr;       // kernels of a search level that nothing on `stream` waits for until a later level (search.cu: k_finalize_terminal)
	cudaEvent_t  ev_fork = nullptr, ev_join = nullptr;
	std::vector<cudaEvent_t> copy_events;     // events of the tickets copy_retired + 1 ... (abw_h2d_async)
	uint64_t     copy_retired = 0;            // tickets retired by abw_ctx_synchronize so far
	int          sm_count = 148;
	uint64_t     launches = 0;
	uint64_t     arena_misses = 0;             // device blocks obtained from the driver (cudaMallocAsync) rather than from the context's cache
	std::string  err;
	// optional per-kernel timing (abw_profile_enable): every launch is bracketed by events and waited for
	bool         profiling = false;
	cudaEvent_t  ev_a = nullptr, ev_b = nullptr;
	std::map<std::string, std::pair<uint64_t, double>> prof;   // kernel -> (launches, total ms)
	// device blocks freed by this context, kept for reuse (see abw_arena_alloc): capacity -> block
	std::multimap<size_t, void*> free_blocks;
	std::map<void*, size_t> block_cap;                         // capacity of every block obtained through the arena, cached or in use
	// pinned staging for small host->device uploads (abw_upload_small), free again after every abw_sync
	unsigned char* h_stage = nullptr;
	size_t stage_cap = 0, stage_used = 0;
	// small device->host results fetched by a kernel into mapped pinned memory instead of through the copy engine (abw_fetch, abw_sync)
	struct Fetch { void* h_dst; const unsigned char* slot; size_t bytes; };
	unsigned char* h_bounce = nullptr;
	size_t bounce_cap = 0, bounce_used = 0;
	std::vector<Fetch> pending;
	// progress words of a running split search, written by the device (mapped pinned memory, search.cu)
	void* h_prog = nullptr;
	// scratch of the one-pass prefix sums (scan_sort.cu): ticket, tile sums, tile prefixes, status words
	void* scan_scratch = nullptr;
	size_t scan_cap = 0;
	uint32_t scan_epoch = 0;
	uint64_t scan_tickets = 0;
	uint32_t* scan_failed = nullptr;          // mapped pinned word: set by a prefix sum whose look-back wait gave up, reported and cleared by abw_sync
};

// Small transfers and the copy engines.  Copies of one direction execute in the order they were issued, whatever their stream: an 8-byte
// cudaMemcpyAsync on the compute stream waits for every bulk copy (read records in, .lrn matrix out) that was enqueued before it on the copy
// stream, and the kernels behind it wait too -- measured: end-to-end step = H2D + resident step + D2H, no overlap at all (DESIGN.md section 5).
// Therefore the small transfers bypass the engines, in both directions through pinned memory and a copy kernel on the context stream:
//  * abw_upload_small (descriptors, job lists, tile tables) copies h_src into the pinned staging area, from where a kernel reads it.  An upload that
//    does not fit, or any upload when the pinned allocation failed, is a cudaMemcpyAsync from h_src.
//  * abw_fetch has a kernel write the result into mapped pinned memory, from where abw_sync (cudaStreamSynchronize + copy-out) hands it to the
//    caller's buffer.
// Every device->host result of an entry point is requested with abw_fetch and every wait on the context stream is abw_sync.  Once abw_sync has drained
// the stream, no copy kernel reads or writes a slot any more, so abw_sync makes the whole staging area and bounce buffer free again; ABW_ENTER
// drops fetch requests an earlier, failed call may have left behind.
// abw_sync also fails (cudaErrorTimeout) when a prefix sum enqueued since the previous abw_sync gave up a look-back wait: its results are wrong.
cudaError_t abw_upload_small(abw_ctx* ctx, void* d_dst, const void* h_src, size_t bytes);
cudaError_t abw_fetch(abw_ctx* ctx, void* h_dst, const void* d_src, size_t bytes);
cudaError_t abw_sync(abw_ctx* ctx);

inline int abw_fail(abw_ctx* ctx, int code, const std::string& msg)
{
	if(ctx)
		ctx->err = msg;
	return code;
}

#define ABW_CUDA(ctx, call)                                                                                          \
	do {                                                                                                             \
		cudaError_t e__ = (call);                                                                                    \
		if(e__ != cudaSuccess) {                                                                                     \
			char b__[512];                                                                                           \
			snprintf(b__, sizeof(b__), "%s:%d: %s failed: %s", __FILE__, __LINE__, #call, cudaGetErrorString(e__));   \
			return abw_fail((ctx), ABW_ERR_CUDA, b__);                                                               \
		}                                                                                                            \
	} while(0)

#define ABW_CHECK(expr)                                                                                              \
	do {                                                                                                             \
		int r__ = (expr);                                                                                            \
		if(r__ != ABW_OK)                                                                                            \
			return r__;                                                                                              \
	} while(0)

// Programmatic dependent launch.  Kernels on the context stream are launched with programmatic stream serialization: the next grid is launched
// while the previous one drains, and its CTAs stop in abw_grid_wait() until the previous grid has completed and its memory is visible.  So every
// __global__ function of the library calls abw_grid_wait() first, before any early return, any read of data an earlier kernel wrote and any global
// store.  The chain is only transitive that way: a grid that returned without waiting would let the grid after it overlap the grid before it.
// (tests/test_pdl_sass.py checks that every kernel of the built library holds the wait.)  In a grid launched without the attribute the wait
// returns at once.  abw_launch_dependents() lets the dependent grid be scheduled once every CTA of this grid has called it or exited; where it
// sits never affects correctness, since the dependent still waits for this whole grid.
__device__ __forceinline__ void abw_grid_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void abw_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// The attribute only relaxes the dependency on the previous operation of the stream when that operation is a kernel, and only as far as that kernel
// allows (launch_dependents or exit).  After a memset, a copy or a cudaStreamWaitEvent (a side-stream join) the launch is ordered as a plain one:
// cudaLaunchAttributeProgrammaticStreamSerialization, CUDA Runtime API, "overlap with the previous kernel in the stream, if that kernel requests
// the overlap".  A kernel of another library on the stream (NCCL, torch) never requests it, so a kernel of ours after it starts once it has
// exited, and still waits for its memory in abw_grid_wait().  Therefore every launch carries the attribute, whatever precedes it.
template <typename... Params, typename... Args>
inline cudaError_t abw_launch_pdl(void (*kernel)(Params...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Args&&... args)
{
	cudaLaunchAttribute attr[1];
	attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
	attr[0].val.programmaticStreamSerializationAllowed = 1;
	cudaLaunchConfig_t cfg = {};
	cfg.gridDim = grid;
	cfg.blockDim = block;
	cfg.dynamicSmemBytes = smem;
	cfg.stream = stream;
	cfg.attrs = attr;
	cfg.numAttrs = 1;
	return cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
}

// every launch goes through this so that abw_kernel_launches() is an honest count.  Profiling brackets each launch with events and waits for it,
// so those launches stay plain: the per-kernel times remain comparable with profiles taken before launches overlapped.
#define ABW_LAUNCH(ctx, kernel, grid, block, smem, ...)                                                              \
	do {                                                                                                             \
		if((ctx)->profiling) {                                                                                       \
			cudaEventRecord((ctx)->ev_a, (ctx)->stream);                                                             \
			kernel<<<(grid), (block), (smem), (ctx)->stream>>>(__VA_ARGS__);                                         \
		}                                                                                                            \
		else                                                                                                         \
			abw_launch_pdl(kernel, (grid), (block), (smem), (ctx)->stream, __VA_ARGS__);                             \
		(ctx)->launches++;                                                                                           \
		ABW_CUDA((ctx), cudaGetLastError());                                                                         \
		if((ctx)->profiling) {                                                                                       \
			float ms__ = 0;                                                                                          \
			cudaEventRecord((ctx)->ev_b, (ctx)->stream);                                                             \
			ABW_CUDA((ctx), cudaEventSynchronize((ctx)->ev_b));                                                      \
			cudaEventElapsedTime(&ms__, (ctx)->ev_a, (ctx)->ev_b);                                                   \
			auto& e__ = (ctx)->prof[#kernel];                                                                        \
			e__.first++;                                                                                             \
			e__.second += ms__;                                                                                      \
		}                                                                                                            \
	} while(0)

// Context whose entry point is executing on this host thread (set by ABW_ENTER).  Device buffers come from a per-context arena: blocks are
// obtained with cudaMallocAsync on the context stream and, when released, cached by the context instead of going back to the driver, so
// that after the first pass of a given shape no entry point pays for cuMemCreate / pool growth (which showed up as sporadic 10-20 ms stalls).
// Every block is only ever used in the order of the context stream, which makes immediate reuse safe.
extern thread_local abw_ctx* abw_tls_ctx;
cudaError_t abw_arena_alloc(abw_ctx* ctx, size_t bytes, void** out);
void abw_arena_free(abw_ctx* ctx, void* p);

// one NVTX range per ABI entry point (named after the function), closed when the entry point returns
struct AbwNvtxRange {
	explicit AbwNvtxRange(const char* name) { nvtxRangePushA(name); }
	~AbwNvtxRange() { nvtxRangePop(); }
};

#define ABW_ENTER(ctx)                                                                                               \
	AbwNvtxRange nvtx_range__(__func__);                                                                             \
	do {                                                                                                             \
		ABW_CUDA((ctx), cudaSetDevice((ctx)->device));                                                               \
		abw_tls_ctx = (ctx);                                                                                         \
		(ctx)->pending.clear();                                                                                      \
		(ctx)->bounce_used = 0;                                                                                      \
	} while(0)

template <typename T>
struct DevBuf {
	T*       p = nullptr;
	size_t   n = 0;
	abw_ctx* owner = nullptr;
	DevBuf() {}
	DevBuf(const DevBuf&) = delete;
	DevBuf& operator=(const DevBuf&) = delete;
	~DevBuf() { release(); }
	void release()
	{
		if(p)
			abw_arena_free(owner, p);
		p = nullptr;
		n = 0;
	}
	cudaError_t alloc(size_t count)
	{
		release();
		n = count;
		owner = abw_tls_ctx;
		return abw_arena_alloc(owner, (count ? count : 1) * sizeof(T), (void**)&p);
	}
};

static inline unsigned int abw_div_up(uint64_t a, uint64_t b) { return (unsigned int)((a + b - 1) / b); }

// ---- decoupled look-back, shared by every one-pass kernel (k_scan_onepass, k_flip_prefix, k_sweep_split_scafs, k_sweep_ss, k_partition2) ----
// A tile publishes its aggregate, walks back over its predecessors until it meets a published inclusive prefix, and publishes its own.
// Published words carry the epoch of the launch (or search level) that wrote them: words of earlier epochs read as empty, so the arrays are not
// cleared between launches.
constexpr uint32_t LB_EMPTY = 0, LB_AGG = 1, LB_PREFIX = 2;
constexpr uint32_t LB_SPIN_LIMIT = 1u << 28;      // a bug must not hang the GPU: give up, flag the error, produce garbage that the host rejects

__device__ __forceinline__ uint32_t ld_volatile_u32(const uint32_t* p) { return *reinterpret_cast<const volatile uint32_t*>(p); }
__device__ __forceinline__ void st_volatile_u32(uint32_t* p, uint32_t v) { *reinterpret_cast<volatile uint32_t*>(p) = v; }
__device__ __forceinline__ unsigned long long ld_volatile_u64(const unsigned long long* p) { return *reinterpret_cast<const volatile unsigned long long*>(p); }
__device__ __forceinline__ void st_volatile_u64(unsigned long long* p, unsigned long long v) { *reinterpret_cast<volatile unsigned long long*>(p) = v; }

// Packed layout: one 64-bit word, payload in bits 0-55, epoch (6 bits) in 56-61, state in 62-63.  One store publishes value and state together.
__device__ __forceinline__ unsigned long long lb_pack(unsigned long long payload, uint32_t st, uint32_t epoch)
{
	return payload | ((unsigned long long)(epoch & 63u) << 56) | ((unsigned long long)st << 62);
}
__device__ __forceinline__ uint32_t lb_packed_state(unsigned long long v, uint32_t epoch)
{
	return (((uint32_t)(v >> 56) & 63u) == (epoch & 63u))? (uint32_t)(v >> 62) : LB_EMPTY;
}

// Split layout: a u32 status word (epoch << 2) | state, the value in a slot of its own.  The writer stores the value (st.cg), then publishes the
// state; the reader, once the walk has seen the states, fences and reads the values with ld.cg (lb_split_value).
__device__ __forceinline__ void lb_split_publish(uint32_t* status, uint32_t st, uint32_t epoch)
{
	__threadfence();
	st_volatile_u32(status, (epoch << 2) | st);
}
__device__ __forceinline__ uint32_t lb_split_state(uint32_t raw, uint32_t epoch) { return ((raw >> 2) == epoch)? (raw & 3u) : LB_EMPTY; }
// value of predecessor i for a sum: its aggregate below the prefix, its inclusive prefix at it, zero where the lane does not take part
template <typename T, typename Slot, typename LdCg>
__device__ __forceinline__ T lb_split_value(uint64_t i, bool take, bool at_prefix, const Slot* aggs, const Slot* prefixes, LdCg ld_cg)
{
	__threadfence();
	T v{};
	if(take)
		v = at_prefix? ld_cg(prefixes + i) : ld_cg(aggs + i);
	return v;
}

// The walk of one warp over the predecessors w-1, w-2, ..., w-npred of tile w (npred > 0), 32 per window: lane l of a window reads the word of
// predecessor i = base - l, so higher lanes are earlier tiles.  Once every predecessor of the window up to its nearest published prefix has
// published, fold(word, i, take, first_prefix) runs on all lanes: first_prefix is the lane of that prefix (32: the window has none and the walk
// goes on), take is true on the lanes that hold a predecessor up to and including it.  Returns false when a wait exceeded LB_SPIN_LIMIT.
template <typename Load, typename State, typename Fold>
__device__ __forceinline__ bool lb_walk(uint64_t w, uint32_t npred, Load load, State state, Fold fold)
{
	const uint32_t lane = threadIdx.x & 31;
	uint64_t base = w - 1;
	uint32_t remaining = npred;
	bool done = false, failed = false;
	while(!done && !failed) {
		const uint32_t cnt = min(32u, remaining);
		decltype(load(base)) v{};
		uint32_t first_prefix, spins = 0;
		while(true) {
			if(lane < cnt)
				v = load(base - lane);
			const uint32_t st = state(v);
			const uint32_t pm = __ballot_sync(0xffffffffu, lane < cnt && st == LB_PREFIX);
			const uint32_t em = __ballot_sync(0xffffffffu, lane < cnt && st == LB_EMPTY);
			first_prefix = pm? (uint32_t)(__ffs(pm) - 1) : 32u;
			const uint32_t need = (first_prefix >= 32u)? 0xFFFFFFFFu : ((2u << first_prefix) - 1u);
			if((em & need) == 0)
				break;
			if(++spins >= LB_SPIN_LIMIT) {
				failed = true;
				break;
			}
		}
		if(failed)
			break;
		fold(v, base - lane, lane < cnt && lane <= first_prefix, first_prefix);
		if(first_prefix < 32u)
			done = true;
		else {
			base -= 32;
			remaining -= 32;
		}
	}
	return !failed;
}

// ---- device-wide primitives implemented in scan_sort.cu -------------------------------------------
// exclusive prefix sum of n uint64 values (in place allowed); d_total (may be null) receives the sum
int abw_exclusive_scan_u64(abw_ctx* ctx, const uint64_t* d_in, uint64_t* d_out, uint64_t n, uint64_t* d_total);
// exclusive prefix sum of uint32 inputs into uint64 outputs
int abw_exclusive_scan_u32_to_u64(abw_ctx* ctx, const uint32_t* d_in, uint64_t* d_out, uint64_t n, uint64_t* d_total);

// Stable LSD radix sort of `batch` independent arrays of n (key, value) pairs each (array b at offset b*stride).
// Only key bits [0, nbits) are examined.  Result is left in (keys, vals); (keys_tmp, vals_tmp) are scratch of the same size.
// Digits are 8, 9 or 10 bits wide, placed only over key bits that actually vary (bits equal in all keys of all arrays are skipped).
int abw_radix_sort_pairs_u64(abw_ctx* ctx, uint64_t* d_keys, uint64_t* d_keys_tmp, uint32_t* d_vals, uint32_t* d_vals_tmp, uint64_t n, uint32_t batch,
                             uint64_t stride, int nbits);
int abw_radix_sort_pairs_u32(abw_ctx* ctx, uint32_t* d_keys, uint32_t* d_keys_tmp, uint32_t* d_vals, uint32_t* d_vals_tmp, uint64_t n, uint32_t batch,
                             uint64_t stride, int nbits);
// the same with the set of key bits that differ between any two keys (OR of all keys ^ AND of all keys) supplied by the caller: no inspection pass
int abw_radix_sort_pairs_u32_varying(abw_ctx* ctx, uint32_t* d_keys, uint32_t* d_keys_tmp, uint32_t* d_vals, uint32_t* d_vals_tmp, uint64_t n, uint32_t batch,
                                     uint64_t stride, unsigned long long varying);
