// Column exchange of the dimension-sharded search over NVLink peer memory (one process per GPU, buffers shared through CUDA IPC).
//
// After the feature stage rank r holds the rows (windows) of its own scaffolds, all 180 + samples columns of them; for the split search rank q needs the
// columns q, q + world, q + 2 world, ... of EVERYBODY's rows (abw_search_set_shard_strided).  abw_scatter_columns_milli does that in one kernel: it reads
// the local rows once (coalesced), turns every value into its integer thousandths (the .lrn values are int(1000 x) / 1000.0, abawaca-build.cpp:603: nothing
// is lost, abw_rows_to_milli) and stores the block of every rank straight into that rank's matrix through the peer mapping -- conversion, column split
// and transfer are one pass, the stores of a tile overlap the loads of the next, and no staging copy exists on either side.  (The NCCL all-to-all it
// replaces moved the same bytes at 124 GB/s between two B200s, after a separate conversion and a separate gather of the strided columns.)
// The receiving side reads its buffer as ABW_LAYOUT_ROWMAJOR_MILLI32 after a barrier the caller provides (any stream-ordered collective of all ranks).
#include "features.cuh"
#include <cstring>
#include <algorithm>

struct abw_peer_group {
	abw_ctx* ctx = nullptr;
	int rank = 0, world = 0;
	std::vector<void*> base;                   // base[q]: rank q's buffer in this process's address space (own pointer for q == rank)
};

namespace {

constexpr int PX_ROWS = 32;                   // rows per tile
constexpr int PX_THREADS = 256;
constexpr int PX_MAXW = 16;                   // ranks

struct PeerDst {
	uint32_t* p[PX_MAXW];                      // rank q's matrix [total rows][cnt(q)], already offset to this step's half of its buffer
};

// windows a scaffold keeps: ScafDpData drops scaffolds with a single datapoint (ScafDpData.cpp:92-93)
__global__ void k_kept_windows(const uint64_t* __restrict__ seg_first, uint32_t nscaf, uint32_t* __restrict__ kept)
{
	abw_grid_wait();
	const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
	if(s < nscaf) {
		const uint64_t c = seg_first[s + 1] - seg_first[s];
		kept[s] = (c >= 2)? (uint32_t)c : 0u;
	}
}

// One CTA per tile of PX_ROWS local rows.  Phase 1: the tile (PX_ROWS x ncols doubles, contiguous when ld == ncols) is read with coalesced loads and kept
// as integers in shared memory.  Phase 2: for every rank q the tile's values of the columns q, q + world, ... form ONE contiguous block of
// PX_ROWS x cnt(q) integers of q's matrix (rows are consecutive, the matrix is row major with cnt(q) columns): written with coalesced stores.
// kept_before != null: local row w (a window of scaffold seg_scaf[w]) goes to row row0 + kept_before[scaffold] + (w - first window of the scaffold) of the
// receivers' matrices, and the rows of scaffolds with a single window go nowhere; null: local row w goes to row row0 + w.
__global__ void __launch_bounds__(PX_THREADS) k_scatter_columns(const double* __restrict__ rows, uint64_t nrows, uint64_t ld, uint32_t ncols, uint32_t world,
                                                                uint64_t row0, const PeerDst dst, int* __restrict__ inexact, const uint32_t* __restrict__ seg_scaf,
                                                                const uint64_t* __restrict__ seg_first, const uint64_t* __restrict__ kept_before)
{
	abw_grid_wait();
	extern __shared__ uint32_t tile[];         // [PX_ROWS][ncols]
	__shared__ unsigned long long dst_row[PX_ROWS];
	__shared__ double milli[1001];             // k / 1000.0 for the k-mer frequencies (k <= 1000): the exactness test without a division per value
	for(uint32_t k = threadIdx.x; k <= 1000; k += PX_THREADS)
		milli[k] = __ddiv_rn((double)k, 1000.0);
	__syncthreads();
	bool bad = false;
	for(uint64_t t0 = (uint64_t)blockIdx.x * PX_ROWS; t0 < nrows; t0 += (uint64_t)gridDim.x * PX_ROWS) {
		const uint32_t nr = (uint32_t)min((uint64_t)PX_ROWS, nrows - t0);
		const uint32_t nval = nr * ncols;
		if(threadIdx.x < nr) {
			unsigned long long d = row0 + t0 + threadIdx.x;
			if(kept_before) {
				const uint32_t sc = seg_scaf[t0 + threadIdx.x];
				const uint64_t f = seg_first[sc];
				d = (seg_first[sc + 1] - f >= 2)? row0 + kept_before[sc] + (t0 + threadIdx.x - f) : ~0ull;
			}
			dst_row[threadIdx.x] = d;
		}
		for(uint32_t i = threadIdx.x; i < nval; i += PX_THREADS) {
			const uint32_t r = i / ncols, c = i - r * ncols;
			const double v = rows[(t0 + r) * ld + c];
			const double k = rint(__dmul_rn(v, 1000.0));
			bool ok = (k >= 0.0) && (k < 2147483000.0) && !(v == 0.0 && signbit(v));
			if(ok)
				ok = (k <= 1000.0)? (milli[(uint32_t)k] == v) : (__ddiv_rn(k, 1000.0) == v);
			tile[i] = ok? (uint32_t)k : 0u;
			bad |= !ok;
		}
		__syncthreads();
		for(uint32_t q = 0; q < world; q++) {
			const uint32_t cnt = (ncols > q)? (ncols - q + world - 1) / world : 0u;
			uint32_t* __restrict__ out = dst.p[q];
			const uint32_t nout = nr * cnt;
			for(uint32_t i = threadIdx.x; i < nout; i += PX_THREADS) {
				const uint32_t r = i / cnt, j = i - r * cnt;
				const unsigned long long d = dst_row[r];
				if(d != ~0ull)
					out[d * cnt + j] = tile[r * ncols + q + j * world];
			}
		}
		__syncthreads();
	}
	if(__syncthreads_or(bad) && threadIdx.x == 0 && inexact)
		atomicAdd(inexact, 1);
}

}  // namespace

extern "C" {

int abw_peer_buffer_create(abw_ctx* ctx, size_t bytes, void** d_buf, unsigned char* handle64)
{
	if(!ctx || !d_buf || !handle64)
		return abw_fail(ctx, ABW_ERR_ARG, "abw_peer_buffer_create: null argument");
	ABW_ENTER(ctx);
	static_assert(sizeof(cudaIpcMemHandle_t) == ABW_IPC_HANDLE_BYTES, "cudaIpcMemHandle_t size");
	*d_buf = nullptr;
	ABW_CUDA(ctx, cudaMalloc(d_buf, bytes? bytes : 256));      // not from the context's pool: only plain allocations can be exported
	cudaIpcMemHandle_t h;
	const cudaError_t e = cudaIpcGetMemHandle(&h, *d_buf);
	if(e != cudaSuccess) {
		cudaGetLastError();
		cudaFree(*d_buf);
		*d_buf = nullptr;
		return abw_fail(ctx, ABW_ERR_UNSUPPORTED, std::string("abw_peer_buffer_create: cudaIpcGetMemHandle failed: ") + cudaGetErrorString(e));
	}
	memcpy(handle64, &h, sizeof(h));
	return ABW_OK;
}

int abw_peer_buffer_destroy(abw_ctx* ctx, void* d_buf)
{
	if(!ctx)
		return ABW_ERR_ARG;
	if(d_buf) {
		cudaSetDevice(ctx->device);
		cudaStreamSynchronize(ctx->stream);
		cudaFree(d_buf);
	}
	return ABW_OK;
}

int abw_peer_group_create(abw_ctx* ctx, void* d_own, const unsigned char* handles, int rank, int world, abw_peer_group** out)
{
	if(!ctx || !d_own || !handles || !out || world < 1 || world > PX_MAXW || rank < 0 || rank >= world)
		return abw_fail(ctx, ABW_ERR_ARG, "abw_peer_group_create: bad argument (at most 16 ranks)");
	ABW_ENTER(ctx);
	abw_peer_group* g = new abw_peer_group();
	g->ctx = ctx; g->rank = rank; g->world = world;
	g->base.assign(world, nullptr);
	for(int q = 0; q < world; q++) {
		if(q == rank) {
			g->base[q] = d_own;
			continue;
		}
		cudaIpcMemHandle_t h;
		memcpy(&h, handles + (size_t)q * ABW_IPC_HANDLE_BYTES, sizeof(h));
		const cudaError_t e = cudaIpcOpenMemHandle(&g->base[q], h, cudaIpcMemLazyEnablePeerAccess);
		if(e != cudaSuccess) {
			cudaGetLastError();
			for(int k = 0; k < q; k++)
				if(k != rank && g->base[k])
					cudaIpcCloseMemHandle(g->base[k]);
			delete g;
			return abw_fail(ctx, ABW_ERR_UNSUPPORTED, std::string("abw_peer_group_create: cudaIpcOpenMemHandle failed: ") + cudaGetErrorString(e));
		}
	}
	*out = g;
	return ABW_OK;
}

void abw_peer_group_destroy(abw_peer_group* g)
{
	if(!g)
		return;
	cudaSetDevice(g->ctx->device);
	cudaStreamSynchronize(g->ctx->stream);
	for(int q = 0; q < g->world; q++)
		if(q != g->rank && g->base[q])
			cudaIpcCloseMemHandle(g->base[q]);
	delete g;
}

int abw_scatter_columns_milli(abw_ctx* ctx, const abw_peer_group* g, const abw_segments* segs, const double* d_rows, uint64_t nrows, uint64_t ld, uint32_t ncols,
                              uint64_t row0, size_t buf_offset_bytes, int32_t* d_inexact)
{
	if(!ctx || !g || (!d_rows && nrows) || ld < ncols || ncols == 0)
		return abw_fail(ctx, ABW_ERR_ARG, "abw_scatter_columns_milli: bad argument");
	if((buf_offset_bytes & 3u) != 0)
		return abw_fail(ctx, ABW_ERR_ARG, "abw_scatter_columns_milli: the offset must be a multiple of 4");
	if(segs && segs->nseg != nrows)
		return abw_fail(ctx, ABW_ERR_ARG, "abw_scatter_columns_milli: the matrix must hold one row per window of the segments");
	ABW_ENTER(ctx);
	if(nrows == 0)
		return ABW_OK;
	// rows of scaffolds with a single window are dropped, as abw_search_create_from_features does: kept windows before every scaffold
	DevBuf<uint32_t> kept;
	DevBuf<uint64_t> kept_before;
	if(segs) {
		ABW_CUDA(ctx, kept.alloc(segs->nscaf));
		ABW_CUDA(ctx, kept_before.alloc((size_t)segs->nscaf + 1));
		ABW_LAUNCH(ctx, k_kept_windows, abw_div_up(segs->nscaf, 256), 256, 0, segs->seg_first.p, segs->nscaf, kept.p);
		ABW_CHECK(abw_exclusive_scan_u32_to_u64(ctx, kept.p, kept_before.p, segs->nscaf, kept_before.p + segs->nscaf));
	}
	const size_t smem = (size_t)PX_ROWS * ncols * sizeof(uint32_t);
	if(smem > 200 * 1024)
		return abw_fail(ctx, ABW_ERR_UNSUPPORTED, "abw_scatter_columns_milli: more than 1600 columns");
	PeerDst dst;
	for(int q = 0; q < PX_MAXW; q++)
		dst.p[q] = (q < g->world)? reinterpret_cast<uint32_t*>((unsigned char*)g->base[q] + buf_offset_bytes) : nullptr;
	if(smem > 48 * 1024)
		ABW_CUDA(ctx, cudaFuncSetAttribute(k_scatter_columns, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
	const unsigned int ctas = (unsigned int)std::min<uint64_t>(abw_div_up(nrows, PX_ROWS), (uint64_t)ctx->sm_count * 8);
	ABW_LAUNCH(ctx, k_scatter_columns, ctas, PX_THREADS, smem, d_rows, nrows, ld, ncols, (uint32_t)g->world, row0, dst, (int*)d_inexact,
	           segs? segs->seg_scaf.p : (const uint32_t*)nullptr, segs? segs->seg_first.p : (const uint64_t*)nullptr, segs? kept_before.p : (const uint64_t*)nullptr);
	return ABW_OK;
}

}  // extern "C"
