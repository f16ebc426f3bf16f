// Assembly in 2 bits per base: abw_pack_2bit decodes UCSC-order codes plus runs of non-ACGT characters into the abw_seqset layout of
// features.cu (see the comment at its top), and the abw_twobit_* entry points read UCSC .2bit files into that form, count their bases
// (k_2bit_base_gc) and write them back as FASTA text (abw_twobit_format, fastaout.cu).
//
// Three kernels, in stream order:
//   k_2bit_decode  one warp per scaffold, 64 bases (16 code bytes) per lane and step: packed words, valid = every position < len, nmask = 0,
//                  C+G count of the decoded codes, countN = 0.
//   k_2bit_runs    one warp per run: clears codes and valid bits under the run, sets nmask bits for N runs (atomics: runs may share words with
//                  neighbouring runs, also runs of another kind), and flags the scaffold.
//   k_2bit_recount one warp per flagged scaffold: countN = popcount(nmask), countGC from the C/G codes.  Non-ACGT positions hold code 0 (A), so
//                  the C/G codes are the C/G bases; counting after the runs makes the counts independent of run order and overlap.
#include "common.cuh"
#include <algorithm>
#include <cctype>
#include <cstring>

#include "features.cuh"
#include "fastaout.cuh"

namespace {

// four bytes of UCSC codes (T=0 C=1 A=2 G=3, first base in the high bits of its byte) -> sixteen internal codes (A=0 C=1 G=2 T=3, base i of the
// word at bits 2i): per 2-bit field hi' = !(hi ^ lo), lo' = !hi, then the four fields of every byte reversed.  Plain integer arithmetic, no table.
__device__ __forceinline__ uint32_t ucsc_to_internal(uint32_t x)
{
	const uint32_t hi = (x >> 1) & 0x55555555u, lo = x & 0x55555555u;
	uint32_t y = (~hi & 0x55555555u) | ((~(hi ^ lo) & 0x55555555u) << 1);
	y = ((y >> 2) & 0x33333333u) | ((y & 0x33333333u) << 2);
	y = ((y >> 4) & 0x0F0F0F0Fu) | ((y & 0x0F0F0F0Fu) << 4);
	return y;
}

// bases with code C (1) or G (2) among the 16 of a packed word: the two bits of the code differ
__device__ __forceinline__ uint32_t gc_of_word(uint32_t w) { return __popc((w ^ (w >> 1)) & 0x55555555u); }

// the low `n` bits set (0 <= n <= 32)
__device__ __forceinline__ uint32_t low_bits(int64_t n) { return n <= 0? 0u : n >= 32? 0xFFFFFFFFu : ((1u << (uint32_t)n) - 1u); }

// 16 bits -> 32 bits, bit i to bits 2i and 2i+1 (a validity mask of 16 bases -> the code bits of a packed word)
__device__ __forceinline__ uint32_t spread2(uint32_t x)
{
	x &= 0xFFFFu;
	x = (x | (x << 8)) & 0x00FF00FFu;
	x = (x | (x << 4)) & 0x0F0F0F0Fu;
	x = (x | (x << 2)) & 0x33333333u;
	x = (x | (x << 1)) & 0x55555555u;
	return x | (x << 1);
}

// One warp per scaffold; a lane takes 16 code bytes (64 bases) per step, read as two aligned 16-byte loads and shifted into place (a scaffold
// may start at any byte), and writes four packed words and two valid / nmask words with one 16-byte and two 8-byte stores.
__global__ void __launch_bounds__(256) k_2bit_decode(const uint8_t* __restrict__ codes, uint64_t nbytes, const uint64_t* __restrict__ byte_off,
                                                     const uint64_t* __restrict__ len, const uint64_t* __restrict__ base, uint32_t nscaf,
                                                     uint32_t* __restrict__ packed, uint32_t* __restrict__ valid, uint32_t* __restrict__ nmask,
                                                     unsigned long long* __restrict__ countN, unsigned long long* __restrict__ countGC)
{
	abw_grid_wait();
	const int lane = threadIdx.x & 31;
	const uint64_t warp0 = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
	for(uint64_t s = warp0; s < nscaf; s += nwarps) {
		const uint64_t L = len[s], b0 = base[s], padded = base[s + 1] - b0, boff = byte_off[s];
		uint32_t nGC = 0;
		for(uint64_t p = 64 * (uint64_t)lane; p < padded; p += 2048) {
			uint32_t w[4] = {0u, 0u, 0u, 0u};
			if(p < L) {
				const uint64_t a = boff + (p >> 2), nb = min((uint64_t)16, (L - p + 3) >> 2);
				const uint64_t al = a & ~15ull;
				if(nb == 16 && al + 32 <= nbytes) {
					const uint4 A = __ldg(reinterpret_cast<const uint4*>(codes + al)), B = __ldg(reinterpret_cast<const uint4*>(codes + al + 16));
					const uint32_t sh = (uint32_t)(a & 15), r8 = (sh & 3u) * 8u;
					switch(sh >> 2) {                           // uniform over the warp: every lane of a scaffold has the same misalignment
					case 0: w[0] = __funnelshift_r(A.x, A.y, r8); w[1] = __funnelshift_r(A.y, A.z, r8); w[2] = __funnelshift_r(A.z, A.w, r8); w[3] = __funnelshift_r(A.w, B.x, r8); break;
					case 1: w[0] = __funnelshift_r(A.y, A.z, r8); w[1] = __funnelshift_r(A.z, A.w, r8); w[2] = __funnelshift_r(A.w, B.x, r8); w[3] = __funnelshift_r(B.x, B.y, r8); break;
					case 2: w[0] = __funnelshift_r(A.z, A.w, r8); w[1] = __funnelshift_r(A.w, B.x, r8); w[2] = __funnelshift_r(B.x, B.y, r8); w[3] = __funnelshift_r(B.y, B.z, r8); break;
					default: w[0] = __funnelshift_r(A.w, B.x, r8); w[1] = __funnelshift_r(B.x, B.y, r8); w[2] = __funnelshift_r(B.y, B.z, r8); w[3] = __funnelshift_r(B.z, B.w, r8); break;
					}
				}
				else {
					// the scaffold's last bytes, or the end of the buffer: only the bytes that belong to the scaffold are read
#pragma unroll
					for(int i = 0; i < 4; i++) {
#pragma unroll
						for(int j = 0; j < 4; j++) {
							const uint32_t k = i * 4 + j;
							if(k < nb)
								w[i] |= (uint32_t)codes[a + k] << (8 * j);
						}
					}
				}
			}
			const int64_t left = (int64_t)L - (int64_t)p;      // bases of the scaffold from p on (may be <= 0 in the padding)
			uint32_t out[4];
#pragma unroll
			for(int i = 0; i < 4; i++) {
				const uint32_t m = low_bits(2 * (left - 16 * i));        // code bits of the positions < L
				out[i] = ucsc_to_internal(w[i]) & m;
				nGC += gc_of_word(out[i]);
			}
			const uint64_t q = b0 + p;                          // a multiple of 64: the stores are aligned
			*reinterpret_cast<uint4*>(packed + (q >> 4)) = make_uint4(out[0], out[1], out[2], out[3]);
			*reinterpret_cast<uint2*>(valid + (q >> 5)) = make_uint2(low_bits(left), low_bits(left - 32));
			*reinterpret_cast<uint2*>(nmask + (q >> 5)) = make_uint2(0u, 0u);
		}
		nGC = __reduce_add_sync(0xffffffffu, nGC);
		if(lane == 0) {
			countN[s] = 0;
			countGC[s] = nGC;
		}
	}
}

// One warp per run, lanes over the 32-base words it touches.  AND / OR are order-independent, so overlapping runs of either kind give the
// same result in any order: a position under an N run is N, under runs of the other kind only is OTHER.
__global__ void __launch_bounds__(256) k_2bit_runs(const abw_base_run* __restrict__ runs, uint64_t nruns, const uint64_t* __restrict__ len,
                                                   const uint64_t* __restrict__ base, uint32_t nscaf, uint32_t* __restrict__ packed,
                                                   uint32_t* __restrict__ valid, uint32_t* __restrict__ nmask, uint32_t* __restrict__ touched)
{
	abw_grid_wait();
	const int lane = threadIdx.x & 31;
	const uint64_t warp0 = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
	for(uint64_t r = warp0; r < nruns; r += nwarps) {
		const abw_base_run run = runs[r];
		if(run.scaf >= nscaf || run.len == 0)
			continue;
		const uint64_t L = len[run.scaf];
		if(run.start >= L)
			continue;
		const uint64_t b0 = base[run.scaf], start = run.start, end = min(start + (uint64_t)run.len, L);
		const bool isN = run.kind == ABW_BASE_N;
		if(lane == 0)
			touched[run.scaf] = 1u;
		for(uint64_t u = (start >> 5) + lane; u <= ((end - 1) >> 5); u += 32) {
			const int64_t lo = (int64_t)start - (int64_t)(u << 5), hi = (int64_t)end - (int64_t)(u << 5);   // [lo, hi) relative to the word
			const uint32_t m = low_bits(hi) & ~low_bits(lo);
			const uint64_t vw = (b0 >> 5) + u;
			atomicAnd(valid + vw, ~m);
			if(isN)
				atomicOr(nmask + vw, m);
			if(m & 0xFFFFu)
				atomicAnd(packed + 2 * vw, ~spread2(m));
			if(m >> 16)
				atomicAnd(packed + 2 * vw + 1, ~spread2(m >> 16));
		}
	}
}

__global__ void __launch_bounds__(256) k_2bit_recount(const uint32_t* __restrict__ touched, const uint64_t* __restrict__ base, uint32_t nscaf,
                                                      const uint32_t* __restrict__ packed, const uint32_t* __restrict__ nmask,
                                                      unsigned long long* __restrict__ countN, unsigned long long* __restrict__ countGC)
{
	abw_grid_wait();
	const int lane = threadIdx.x & 31;
	const uint64_t warp0 = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
	for(uint64_t s = warp0; s < nscaf; s += nwarps) {
		if(!touched[s])
			continue;
		const uint64_t b0 = base[s], padded = base[s + 1] - b0;     // bits past the length are 0 in both arrays
		uint32_t nN = 0, nGC = 0;
		for(uint64_t u = lane; u < (padded >> 5); u += 32) {
			const uint64_t vw = (b0 >> 5) + u;
			nN += __popc(nmask[vw]);
			nGC += gc_of_word(packed[2 * vw]) + gc_of_word(packed[2 * vw + 1]);
		}
		nN = __reduce_add_sync(0xffffffffu, nN);
		nGC = __reduce_add_sync(0xffffffffu, nGC);
		if(lane == 0) {
			countN[s] = nN;
			countGC[s] = nGC;
		}
	}
}

// One warp per record of a .2bit file: C+G = the C/G codes (UCSC C = 1, G = 3: the low bit) of its bases, less those under its N blocks.
__global__ void __launch_bounds__(256) k_2bit_base_gc(const uint8_t* __restrict__ file, const uint64_t* __restrict__ dna_off, const uint64_t* __restrict__ len,
                                                      const uint64_t* __restrict__ nblk0, const uint2* __restrict__ nblocks, uint64_t nrec,
                                                      unsigned long long* __restrict__ countGC)
{
	abw_grid_wait();
	const int lane = threadIdx.x & 31;
	const uint64_t warp0 = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
	for(uint64_t r = warp0; r < nrec; r += nwarps) {
		const uint64_t L = len[r];
		const uint8_t* __restrict__ dna = file + dna_off[r];
		int64_t nGC = 0;
		for(uint64_t i = lane; i < (L + 3) >> 2; i += 32) {
			const uint32_t keep = (4 * i + 4 <= L)? 0xFFu : (0xFFu << (2 * (4 * i + 4 - L))) & 0xFFu;      // codes of bases past L are padding
			nGC += __popc((uint32_t)dna[i] & keep & 0x55u);
		}
		for(uint64_t k = nblk0[r]; k < nblk0[r + 1]; k++) {
			const uint2 nb = nblocks[k];
			for(uint64_t p = (uint64_t)nb.x + lane; p < (uint64_t)nb.x + nb.y; p += 32)
				nGC -= (dna[p >> 2] >> (6 - 2 * (p & 3))) & 1u;
		}
		for(int o = 16; o > 0; o >>= 1)
			nGC += __shfl_down_sync(0xffffffffu, nGC, o);
		if(lane == 0)
			countGC[r] = (unsigned long long)nGC;
	}
}

int pack_2bit_impl(abw_ctx* ctx, abw_seqset* s, const abw_2bit_assembly* in, uint32_t nscaf)
{
	s->nscaf = nscaf;
	s->h_len.resize(nscaf);
	s->h_base.resize((size_t)nscaf + 1);
	uint64_t b = 0;
	for(uint32_t i = 0; i < nscaf; i++) {
		const uint64_t L = in->h_len[i];
		if(L >= (1ull << 32))
			return abw_fail(ctx, ABW_ERR_ARG, "abw_pack_2bit: a scaffold length must be below 2^32");
		if(in->h_byte_off[i] > in->nbytes || (L + 3) / 4 > in->nbytes - in->h_byte_off[i])
			return abw_fail(ctx, ABW_ERR_ARG, "abw_pack_2bit: a scaffold's codes reach past the end of the code buffer");
		s->h_len[i] = L;
		s->h_base[i] = b;
		b += (L + 127) & ~127ull;
	}
	s->h_base[nscaf] = b;
	s->total_padded = b;
	DevBuf<uint64_t> d_boff;
	DevBuf<uint32_t> touched;
	ABW_CUDA(ctx, d_boff.alloc(nscaf));
	ABW_CUDA(ctx, abw_upload_small(ctx, d_boff.p, in->h_byte_off, sizeof(uint64_t) * nscaf));
	ABW_CUDA(ctx, s->len.alloc(nscaf));
	ABW_CUDA(ctx, s->base.alloc((size_t)nscaf + 1));
	ABW_CUDA(ctx, abw_upload_small(ctx, s->len.p, s->h_len.data(), sizeof(uint64_t) * nscaf));
	ABW_CUDA(ctx, abw_upload_small(ctx, s->base.p, s->h_base.data(), sizeof(uint64_t) * ((size_t)nscaf + 1)));
	// + slack so that the k-mer kernel may read one word past a segment (as pack_impl in features.cu)
	ABW_CUDA(ctx, s->packed.alloc(b / 16 + 16));
	ABW_CUDA(ctx, s->valid.alloc(b / 32 + 16));
	ABW_CUDA(ctx, s->nmask.alloc(b / 32 + 16));
	ABW_CUDA(ctx, cudaMemsetAsync(s->packed.p + b / 16, 0, 16 * sizeof(uint32_t), ctx->stream));
	ABW_CUDA(ctx, cudaMemsetAsync(s->valid.p + b / 32, 0, 16 * sizeof(uint32_t), ctx->stream));
	ABW_CUDA(ctx, cudaMemsetAsync(s->nmask.p + b / 32, 0, 16 * sizeof(uint32_t), ctx->stream));
	ABW_CUDA(ctx, s->countN.alloc(nscaf));
	ABW_CUDA(ctx, s->countGC.alloc(nscaf));
	ABW_CHECK(abw_wait_h2d(ctx, in->h2d_ticket));                  // on the device: codes and runs may still be on their way
	if(nscaf == 0)
		return ABW_OK;
	const unsigned int blocks = (unsigned int)std::min<uint64_t>(abw_div_up((uint64_t)nscaf * 32, 256), (uint64_t)ctx->sm_count * 16);
	ABW_LAUNCH(ctx, k_2bit_decode, blocks, 256, 0, in->codes, in->nbytes, d_boff.p, s->len.p, s->base.p, nscaf, s->packed.p, s->valid.p, s->nmask.p,
	           s->countN.p, s->countGC.p);
	if(in->nruns > 0) {
		ABW_CUDA(ctx, touched.alloc(nscaf));
		ABW_CUDA(ctx, cudaMemsetAsync(touched.p, 0, sizeof(uint32_t) * nscaf, ctx->stream));
		const unsigned int rblocks = (unsigned int)std::min<uint64_t>(abw_div_up(in->nruns * 32, 256), (uint64_t)ctx->sm_count * 16);
		ABW_LAUNCH(ctx, k_2bit_runs, rblocks, 256, 0, in->runs, in->nruns, s->len.p, s->base.p, nscaf, s->packed.p, s->valid.p, s->nmask.p, touched.p);
		ABW_LAUNCH(ctx, k_2bit_recount, blocks, 256, 0, touched.p, s->base.p, nscaf, s->packed.p, s->nmask.p, s->countN.p, s->countGC.p);
	}
	return ABW_OK;
}

// ---------------------------------------------------------------------------------------------------
// UCSC .2bit: header {signature, version, sequence count, reserved}, index {name size (1 byte), name, offset (4 bytes in version 0, 8 in 1)},
// per record {DNA size, N block count, N starts, N sizes, mask block count, mask starts, mask sizes, reserved, packed DNA}, all words in the
// byte order the signature shows.
// ---------------------------------------------------------------------------------------------------
constexpr uint32_t TWOBIT_SIG = 0x1A412743u;

struct Block { uint32_t start, size; };

}  // namespace

struct abw_twobit {
	uint64_t nbytes = 0;
	std::vector<uint64_t> name_off, seq_len, dna_off;
	std::vector<uint32_t> name_len;
	std::vector<uint64_t> nblk0, mblk0;      // [nrec + 1]: the record's blocks in nblocks / mblocks
	std::vector<Block> nblocks, mblocks;
	DevBuf<uint2> d_nblocks;                 // nblocks on the device {start, size}, for abw_twobit_format / abw_twobit_base_counts
};

namespace {

struct Reader {
	const uint8_t* p;
	uint64_t n;
	bool swap;
	bool ok = true;
	uint64_t u32(uint64_t at)
	{
		if(at > n || n - at < 4) { ok = false; return 0; }
		uint32_t v;
		memcpy(&v, p + at, 4);
		return swap? __builtin_bswap32(v) : v;
	}
	uint64_t u64(uint64_t at)
	{
		if(at > n || n - at < 8) { ok = false; return 0; }
		uint64_t v;
		memcpy(&v, p + at, 8);
		return swap? __builtin_bswap64(v) : v;
	}
};

// count blocks at `at` (starts, then sizes): inside [0, L), sorted, not overlapping
bool read_blocks(Reader& R, uint64_t& at, uint64_t L, std::vector<Block>& out)
{
	const uint64_t count = R.u32(at);
	at += 4;
	if(!R.ok || count > (R.n - std::min(at, R.n)) / 8)
		return false;
	uint64_t prev_end = 0;
	for(uint64_t i = 0; i < count; i++) {
		const uint64_t st = R.u32(at + 4 * i), sz = R.u32(at + 4 * count + 4 * i);
		if(st < prev_end || st + sz > L)
			return false;
		prev_end = st + sz;
		out.push_back(Block{(uint32_t)st, (uint32_t)sz});
	}
	at += 8 * count;
	return R.ok;
}

int twobit_scan_impl(abw_ctx* ctx, abw_twobit* t, const uint8_t* f, uint64_t nbytes)
{
	auto bad = [&](const char* what) { return abw_fail(ctx, ABW_ERR_ARG, std::string("abw_twobit_scan: ") + what); };
	if(nbytes < 16)
		return bad("truncated header");
	uint32_t sig;
	memcpy(&sig, f, 4);
	Reader R{f, nbytes, false};
	if(sig == __builtin_bswap32(TWOBIT_SIG))
		R.swap = true;
	else if(sig != TWOBIT_SIG)
		return bad("not a .2bit file (signature)");
	const uint64_t version = R.u32(4), count = R.u32(8);
	if(version > 1)
		return bad("unknown version");
	const uint64_t osz = version? 8 : 4;
	t->nbytes = nbytes;
	t->nblk0.push_back(0);
	t->mblk0.push_back(0);
	uint64_t at = 16;
	for(uint64_t i = 0; i < count; i++) {
		if(at >= nbytes)
			return bad("truncated index");
		const uint64_t nl = f[at];
		if(nl == 0)
			return bad("empty name");
		if(nbytes - at - 1 < nl + osz)
			return bad("truncated index");
		t->name_off.push_back(at + 1);
		t->name_len.push_back((uint32_t)nl);
		const uint64_t off = version? R.u64(at + 1 + nl) : R.u32(at + 1 + nl);
		at += 1 + nl + osz;
		uint64_t r = off;
		const uint64_t L = R.u32(r);
		r += 4;
		if(!R.ok)
			return bad("record offset outside the file");
		if(!read_blocks(R, r, L, t->nblocks))
			return bad("N blocks outside the file or the sequence, unsorted or overlapping");
		if(!read_blocks(R, r, L, t->mblocks))
			return bad("mask blocks outside the file or the sequence, unsorted or overlapping");
		r += 4;                                              // reserved
		if(r > nbytes || (L + 3) / 4 > nbytes - r)
			return bad("packed DNA outside the file");
		t->seq_len.push_back(L);
		t->dna_off.push_back(r);
		t->nblk0.push_back(t->nblocks.size());
		t->mblk0.push_back(t->mblocks.size());
	}
	return ABW_OK;
}

}  // namespace

// ===================================================================================================
// C ABI
// ===================================================================================================
extern "C" {

int abw_pack_2bit(abw_ctx* ctx, const abw_2bit_assembly* in, uint32_t nscaf, abw_seqset** out)
{
	if(!ctx || !in || !out || (nscaf && (!in->h_byte_off || !in->h_len)) || (!in->codes && in->nbytes) || (!in->runs && in->nruns))
		return abw_fail(ctx, ABW_ERR_ARG, "abw_pack_2bit: null argument");
	ABW_ENTER(ctx);
	abw_seqset* s = new abw_seqset();
	int rc = pack_2bit_impl(ctx, s, in, nscaf);
	if(rc != ABW_OK) {
		delete s;
		return rc;
	}
	*out = s;
	return ABW_OK;
}

int abw_twobit_scan(abw_ctx* ctx, const void* h_file, uint64_t nbytes, abw_twobit** out)
{
	if(!ctx || !out || (!h_file && nbytes))
		return abw_fail(ctx, ABW_ERR_ARG, "abw_twobit_scan: null argument");
	ABW_ENTER(ctx);
	abw_twobit* t = new abw_twobit();
	int rc = twobit_scan_impl(ctx, t, (const uint8_t*)h_file, nbytes);
	if(rc == ABW_OK && !t->nblocks.empty()) {
		static_assert(sizeof(Block) == sizeof(uint2), "N blocks go to the device as uint2");
		const cudaError_t e = t->d_nblocks.alloc(t->nblocks.size());
		if(e == cudaSuccess)
			rc = abw_upload_small(ctx, t->d_nblocks.p, t->nblocks.data(), sizeof(Block) * t->nblocks.size()) == cudaSuccess? ABW_OK : ABW_ERR_CUDA;
		else
			rc = ABW_ERR_CUDA;
		if(rc != ABW_OK)
			abw_fail(ctx, rc, "abw_twobit_scan: could not copy the N blocks to the device");
	}
	if(rc != ABW_OK) {
		delete t;
		return rc;
	}
	*out = t;
	return ABW_OK;
}

void abw_twobit_destroy(abw_twobit* t) { delete t; }

uint64_t abw_twobit_count(const abw_twobit* t) { return t? t->seq_len.size() : 0; }

int abw_twobit_get(abw_ctx* ctx, const abw_twobit* t, uint64_t* h_name_off, uint32_t* h_name_len, uint64_t* h_seq_len)
{
	if(!ctx || !t)
		return abw_fail(ctx, ABW_ERR_ARG, "abw_twobit_get: null argument");
	const size_t n = t->seq_len.size();
	if(h_name_off && n)
		memcpy(h_name_off, t->name_off.data(), sizeof(uint64_t) * n);
	if(h_name_len && n)
		memcpy(h_name_len, t->name_len.data(), sizeof(uint32_t) * n);
	if(h_seq_len && n)
		memcpy(h_seq_len, t->seq_len.data(), sizeof(uint64_t) * n);
	return ABW_OK;
}

int abw_twobit_decode(abw_ctx* ctx, const abw_twobit* t, uint64_t record, const void* h_file, char* h_out)
{
	if(!ctx || !t || !h_file || (!h_out && record < t->seq_len.size() && t->seq_len[record]))
		return abw_fail(ctx, ABW_ERR_ARG, "abw_twobit_decode: null argument");
	if(record >= t->seq_len.size())
		return abw_fail(ctx, ABW_ERR_ARG, "abw_twobit_decode: record index out of range");
	const uint8_t* dna = (const uint8_t*)h_file + t->dna_off[record];
	const uint64_t L = t->seq_len[record];
	for(uint64_t i = 0; i < L; i++)
		h_out[i] = "TCAG"[(dna[i >> 2] >> (6 - 2 * (i & 3))) & 3];
	for(uint64_t k = t->nblk0[record]; k < t->nblk0[record + 1]; k++)
		memset(h_out + t->nblocks[k].start, 'N', t->nblocks[k].size);
	for(uint64_t k = t->mblk0[record]; k < t->mblk0[record + 1]; k++)
		for(uint64_t i = t->mblocks[k].start; i < (uint64_t)t->mblocks[k].start + t->mblocks[k].size; i++)
			h_out[i] = (char)tolower((unsigned char)h_out[i]);
	return ABW_OK;
}

int abw_twobit_pack(abw_ctx* ctx, const abw_twobit* t, const void* d_file, uint64_t h2d_ticket, const uint32_t* h_order, uint32_t nout, abw_seqset** out)
{
	if(!ctx || !t || !out || (!h_order && nout) || (!d_file && t->nbytes))
		return abw_fail(ctx, ABW_ERR_ARG, "abw_twobit_pack: null argument");
	ABW_ENTER(ctx);
	const uint64_t nrec = t->seq_len.size();
	std::vector<uint64_t> byte_off(nout), lens(nout);
	std::vector<abw_base_run> runs;
	std::vector<uint8_t> used(nrec, 0);
	for(uint32_t i = 0; i < nout; i++) {
		const uint64_t r = h_order[i];
		if(r >= nrec)
			return abw_fail(ctx, ABW_ERR_ARG, "abw_twobit_pack: record index out of range");
		if(used[r])
			return abw_fail(ctx, ABW_ERR_ARG, "abw_twobit_pack: a record may appear only once in the order");
		used[r] = 1;
		byte_off[i] = t->dna_off[r];
		lens[i] = t->seq_len[r];
		// both block lists are sorted and disjoint: one merge finds an N block under a mask block
		uint64_t m = t->mblk0[r];
		for(uint64_t k = t->nblk0[r]; k < t->nblk0[r + 1]; k++) {
			const Block nb = t->nblocks[k];
			if(nb.size == 0)
				continue;
			while(m < t->mblk0[r + 1] && (uint64_t)t->mblocks[m].start + t->mblocks[m].size <= nb.start)
				m++;
			for(uint64_t j = m; j < t->mblk0[r + 1] && t->mblocks[j].start < (uint64_t)nb.start + nb.size; j++)
				if(t->mblocks[j].size > 0)
					return abw_fail(ctx, ABW_ERR_ILLEGAL_DNA, "Illegal_DNAString: lower-case 'n' in a sequence (an N block under a mask block, String.cpp:47-49)");
			runs.push_back(abw_base_run{i, nb.start, nb.size, ABW_BASE_N});
		}
	}
	DevBuf<abw_base_run> d_runs;
	if(!runs.empty()) {
		ABW_CUDA(ctx, d_runs.alloc(runs.size()));
		ABW_CUDA(ctx, abw_upload_small(ctx, d_runs.p, runs.data(), sizeof(abw_base_run) * runs.size()));
	}
	abw_2bit_assembly in;
	in.codes = (const uint8_t*)d_file;
	in.nbytes = t->nbytes;
	in.h_byte_off = byte_off.data();
	in.h_len = lens.data();
	in.runs = d_runs.p;
	in.nruns = runs.size();
	in.h2d_ticket = h2d_ticket;
	abw_seqset* s = new abw_seqset();
	int rc = pack_2bit_impl(ctx, s, &in, nout);
	if(rc != ABW_OK) {
		delete s;
		return rc;
	}
	*out = s;
	return ABW_OK;
}

int abw_twobit_format(abw_ctx* ctx, const abw_twobit* t, const void* d_file, uint64_t h2d_ticket, const uint32_t* h_recs, uint64_t nrecs, uint64_t byte0, char* d_text,
                      uint64_t cap, uint64_t* total_bytes, uint64_t* nbytes)
{
	if(!ctx || !t || !total_bytes || !nbytes || (!h_recs && nrecs) || (!d_file && t->nbytes))
		return abw_fail(ctx, ABW_ERR_ARG, "abw_twobit_format: null argument");
	ABW_ENTER(ctx);
	*total_bytes = 0;
	*nbytes = 0;
	const uint64_t nrec = t->seq_len.size();
	std::vector<FaRecord> recs(nrecs);
	for(uint64_t i = 0; i < nrecs; i++) {
		const uint32_t r = h_recs[i];
		if(r >= nrec)
			return abw_fail(ctx, ABW_ERR_ARG, "abw_twobit_format: record index out of range");
		recs[i] = FaRecord{t->name_off[r], 0, t->dna_off[r], t->seq_len[r], t->nblk0[r], t->nblk0[r + 1], t->name_len[r], 0};
	}
	ABW_CHECK(abw_wait_h2d(ctx, h2d_ticket));                      // on the device: the file image may still be on its way
	FaSource src;
	src.kind = FA_SRC_2BIT;
	src.text = (const char*)d_file;
	src.nblocks = t->d_nblocks.p;
	return abw_fasta_text(ctx, src, recs, byte0, d_text, cap, total_bytes, nbytes);
}

int abw_twobit_base_counts(abw_ctx* ctx, const abw_twobit* t, const void* d_file, uint64_t h2d_ticket, uint64_t* h_count_N, uint64_t* h_count_GC)
{
	const uint64_t nrec = t? t->seq_len.size() : 0;
	if(!ctx || !t || ((!h_count_N || !h_count_GC) && nrec) || (!d_file && t->nbytes))
		return abw_fail(ctx, ABW_ERR_ARG, "abw_twobit_base_counts: null argument");
	ABW_ENTER(ctx);
	ABW_CHECK(abw_wait_h2d(ctx, h2d_ticket));
	if(nrec == 0)
		return ABW_OK;
	DevBuf<uint64_t> d_off, d_len, d_blk0;
	DevBuf<unsigned long long> d_gc;
	ABW_CUDA(ctx, d_off.alloc(nrec));
	ABW_CUDA(ctx, d_len.alloc(nrec));
	ABW_CUDA(ctx, d_blk0.alloc(nrec + 1));
	ABW_CUDA(ctx, d_gc.alloc(nrec));
	ABW_CUDA(ctx, abw_upload_small(ctx, d_off.p, t->dna_off.data(), sizeof(uint64_t) * nrec));
	ABW_CUDA(ctx, abw_upload_small(ctx, d_len.p, t->seq_len.data(), sizeof(uint64_t) * nrec));
	ABW_CUDA(ctx, abw_upload_small(ctx, d_blk0.p, t->nblk0.data(), sizeof(uint64_t) * (nrec + 1)));
	const unsigned int blocks = (unsigned int)std::min<uint64_t>(abw_div_up(nrec * 32, 256), (uint64_t)ctx->sm_count * 16);
	ABW_LAUNCH(ctx, k_2bit_base_gc, blocks, 256, 0, (const uint8_t*)d_file, d_off.p, d_len.p, d_blk0.p, t->d_nblocks.p, nrec, d_gc.p);
	ABW_CUDA(ctx, abw_fetch(ctx, h_count_GC, d_gc.p, sizeof(uint64_t) * nrec));
	ABW_CUDA(ctx, abw_sync(ctx));
	// N: the sizes of the N blocks, a mask over them or not
	for(uint64_t r = 0; r < nrec; r++) {
		uint64_t n = 0;
		for(uint64_t k = t->nblk0[r]; k < t->nblk0[r + 1]; k++)
			n += t->nblocks[k].size;
		h_count_N[r] = n;
	}
	return ABW_OK;
}

}  // extern "C"
