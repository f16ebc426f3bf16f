// Matrix -> .lrn data lines on the device (SURVEY.md section 8f, row 2: the text writers of abawaca-build and abawaca).
//
// Replaces the per-value printf of
//   abawaca-build.cpp:603           "\t%.3lf" per value of abawaca.lrn
//   ClusterWriter.cpp:81-98         "\t%lf" per value of clusters/<id>.lrn
// Every value is byte-identical to what glibc's printf writes.  A finite double x = m 2^e (m < 2^53) is printed with p decimals from the
// integer N = round(m 10^p 2^e), ties to even: m 10^p < 2^73 fits 128 bits, so the shift by -e leaves the integer part and the remainder exactly
// and the remainder is compared with one half.  That covers |N| < 2^64 (|x| < 1.8e16 with three decimals, 1.8e13 with six); the rest
// (larger magnitudes, inf, nan) is printed by the host's C library and the strings are looked up by the writer.
//
// Data flow: one warp per line computes the line's length (digit counts need no formatting); a one-pass scan gives every line its offset;
// one thread cuts at the caller's capacity; one warp per line formats 32 values at a time in registers, stages the bytes in shared memory at
// the alignment they have in the output and stores them as 16-byte words.
#include "common.cuh"
#include <algorithm>
#include <cstring>
#include <vector>

namespace {

constexpr int TX_WARPS = 8;                        // warps per block; each owns a staging buffer
constexpr int TX_BUF = 4096 + 16;                  // bytes of a warp's buffer: 4 KB of text at the output's alignment mod 16
constexpr uint32_t TX_MAX_COLS = 1u << 22;         // line lengths are 32-bit: 2^22 values of at most 318 bytes (with their tab) stay below 2^31

struct TxFallback { uint64_t key; double v; };     // key = line * ncols + column, line relative to the call

template <int P> struct Pow10;
template <> struct Pow10<3> { static constexpr uint64_t v = 1000ull; };
template <> struct Pow10<6> { static constexpr uint64_t v = 1000000ull; };

// x -> sign, integer part and P-digit fraction of "%.<P>f" (round to nearest, ties to even, as glibc); false: not on the exact integer path
template <int P>
__device__ __forceinline__ bool tx_split(double x, bool& neg, uint64_t& ip, uint32_t& fp)
{
	const uint64_t b = (uint64_t)__double_as_longlong(x);
	neg = (b >> 63) != 0;
	const uint32_t ex = (uint32_t)(b >> 52) & 0x7FFu;
	if(ex == 0x7FFu)
		return false;                                                   // inf, nan
	uint64_t m = b & ((1ull << 52) - 1);
	int e = -1074;                                                      // subnormal (and zero)
	if(ex) {
		m |= 1ull << 52;
		e = (int)ex - 1075;
	}
	const unsigned __int128 t = (unsigned __int128)m * Pow10<P>::v;    // < 2^73
	unsigned __int128 n = 0;
	if(e >= 0) {
		if(e > 11)
			return false;                                               // m >= 2^52: N >= 2^64
		n = t << e;
	}
	else if(-e <= 80) {                                                 // beyond that t < 2^73 <= half a unit: N = 0
		const int s = -e;
		const unsigned __int128 one = 1;
		n = t >> s;
		const unsigned __int128 rem = t & ((one << s) - 1), half = one << (s - 1);
		if(rem > half || (rem == half && (n & 1)))
			n += 1;
	}
	if((uint64_t)(n >> 64))
		return false;
	const uint64_t n64 = (uint64_t)n;
	ip = n64 / Pow10<P>::v;
	fp = (uint32_t)(n64 - ip * Pow10<P>::v);
	return true;
}

__device__ __forceinline__ uint32_t tx_ndigits(uint64_t v)
{
	uint32_t d = 1;
	while(v >= 10) {
		v /= 10;
		d++;
	}
	return d;
}

__device__ __forceinline__ uint64_t tx_row(const uint64_t* __restrict__ rows, uint64_t line0, uint64_t i)
{
	return rows? rows[i] : line0 + i;
}

// length of every line; values off the integer path are listed in fb (their text length is added once the host has printed them)
template <int P>
__global__ void __launch_bounds__(TX_WARPS * 32) k_lrn_text_len(const double* __restrict__ vals, uint64_t ld, uint32_t col0, uint32_t ncols,
                                                               const uint64_t* __restrict__ rows, uint64_t line0, uint64_t nlines,
                                                               uint32_t* __restrict__ line_len, TxFallback* __restrict__ fb, uint32_t fb_cap,
                                                               uint32_t* __restrict__ fb_count)
{
	abw_grid_wait();
	const int lane = threadIdx.x & 31;
	const uint64_t nwarps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
	for(uint64_t i = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; i < nlines; i += nwarps) {
		const uint64_t r = tx_row(rows, line0, i);
		const double* __restrict__ v = vals + r * ld + col0;
		uint32_t len = 0;
		for(uint32_t c = lane; c < ncols; c += 32) {
			bool neg;
			uint64_t ip;
			uint32_t fp;
			const double x = v[c];
			if(tx_split<P>(x, neg, ip, fp))
				len += 1 + (uint32_t)neg + tx_ndigits(ip) + 1 + P;       // tab, sign, integer part, point, fraction
			else {
				len += 1;
				const uint32_t k = atomicAdd(fb_count, 1u);
				if(k < fb_cap) {
					fb[k].key = i * ncols + c;
					fb[k].v = x;
				}
			}
		}
		len = __reduce_add_sync(0xffffffffu, len);
		if(lane == 0)
			line_len[i] = len + tx_ndigits(r + 1) + 1;                   // key and newline
	}
}

__global__ void k_lrn_text_fb_len(const uint64_t* __restrict__ fb_key, const uint32_t* __restrict__ fb_len, uint32_t nfb, uint32_t ncols, uint32_t* __restrict__ line_len)
{
	abw_grid_wait();
	const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
	if(k < nfb)
		atomicAdd(&line_len[fb_key[k] / ncols], fb_len[k]);
}

// cut[0] = whole lines that fit cap bytes, cut[1] = their bytes, cut[2] = bytes of line 0
__global__ void k_lrn_text_cut(const uint64_t* __restrict__ offs, const uint64_t* __restrict__ total, uint64_t nlines, uint64_t cap, uint64_t* __restrict__ cut)
{
	abw_grid_wait();
	const uint64_t tot = *total;
	auto end_of = [&](uint64_t k) { return k + 1 < nlines? offs[k + 1] : tot; };      // end of line k
	uint64_t lo = 0, hi = nlines;                                                       // lines [0, lo) fit; lines [0, hi + 1) do not
	while(lo < hi) {
		const uint64_t mid = lo + (hi - lo + 1) / 2;
		if(end_of(mid - 1) <= cap)
			lo = mid;
		else
			hi = mid - 1;
	}
	cut[0] = lo;
	cut[1] = lo? end_of(lo - 1) : 0;
	cut[2] = end_of(0);
}

// bytes out[a, a + n), staged at buf[address of out + a, mod 16 ...]: 16-byte words where the ADDRESS is aligned (the caller's text buffer may
// start anywhere), single bytes at both ends
__device__ __forceinline__ void tx_flush(const unsigned char* buf, char* __restrict__ out, uint64_t a, uint32_t n, int lane)
{
	__syncwarp();
	const uintptr_t p = reinterpret_cast<uintptr_t>(out + a), e = p + n, base = p & ~(uintptr_t)15;
	const uintptr_t up = (p + 15) & ~(uintptr_t)15, A0 = up < e? up : e, A1 = A0 > (e & ~(uintptr_t)15)? A0 : (e & ~(uintptr_t)15);
	if(lane < (int)(A0 - p))
		reinterpret_cast<char*>(p)[lane] = (char)buf[p + lane - base];
	for(uintptr_t g = A0 + 16 * (uintptr_t)lane; g < A1; g += 16 * 32)
		*reinterpret_cast<uint4*>(g) = *reinterpret_cast<const uint4*>(buf + (g - base));
	if(lane < (int)(e - A1))
		reinterpret_cast<char*>(A1)[lane] = (char)buf[A1 + lane - base];
	__syncwarp();
}

// item = tab + value at dst[0 ..): the integer path, or the host's text of the value
template <int P>
__device__ __forceinline__ void tx_put(unsigned char* dst, bool fast, bool neg, uint64_t ip, uint32_t fp, uint32_t len, const char* __restrict__ fb_text)
{
	dst[0] = '\t';
	if(!fast) {
		for(uint32_t j = 1; j < len; j++)
			dst[j] = (unsigned char)fb_text[j - 1];
		return;
	}
	uint32_t w = len;
	for(int j = 0; j < P; j++) {
		dst[--w] = (unsigned char)('0' + fp % 10);
		fp /= 10;
	}
	dst[--w] = '.';
	do {
		dst[--w] = (unsigned char)('0' + ip % 10);
		ip /= 10;
	} while(ip);
	if(neg)
		dst[--w] = '-';
}

// at least 4 resident blocks: ptxas otherwise holds the kernel to 40 registers and spills
template <int P>
__global__ void __launch_bounds__(TX_WARPS * 32, 4) k_lrn_text_write(const double* __restrict__ vals, uint64_t ld, uint32_t col0, uint32_t ncols,
                                                                 const uint64_t* __restrict__ rows, uint64_t line0, const uint64_t* __restrict__ cut,
                                                                 const uint64_t* __restrict__ offs, const uint64_t* __restrict__ fb_key,
                                                                 const uint64_t* __restrict__ fb_off, const uint32_t* __restrict__ fb_len, uint32_t nfb,
                                                                 const char* __restrict__ fb_text, char* __restrict__ out)
{
	abw_grid_wait();
	__shared__ __align__(16) unsigned char smem[TX_WARPS][TX_BUF];
	const int lane = threadIdx.x & 31;
	unsigned char* buf = smem[threadIdx.x >> 5];
	const uint64_t nlines = cut[0];
	const uint64_t nwarps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
	const uint64_t mis = reinterpret_cast<uintptr_t>(out) & 15;        // staging follows the address of the output, not its offset
	for(uint64_t i = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; i < nlines; i += nwarps) {
		const uint64_t r = tx_row(rows, line0, i);
		const double* __restrict__ v = vals + r * ld + col0;
		uint64_t a = offs[i];                                           // output offset of buf[(a + mis) & 15]
		uint32_t n = 0;                                                 // bytes staged
		{
			uint64_t k = r + 1;
			const uint32_t kd = tx_ndigits(k);
			if(lane == 0)
				for(uint32_t w = kd; w-- > 0; k /= 10)
					buf[((a + mis) & 15) + w] = (unsigned char)('0' + k % 10);
			n = kd;
		}
		for(uint32_t c0 = 0; c0 < ncols; c0 += 32) {
			const uint32_t c = c0 + lane;
			bool neg = false, fast = true;
			uint64_t ip = 0;
			uint32_t fp = 0, len = 0;
			const char* ft = nullptr;
			if(c < ncols) {
				fast = tx_split<P>(v[c], neg, ip, fp);
				if(fast)
					len = 1 + (uint32_t)neg + tx_ndigits(ip) + 1 + P;
				else {
					const uint64_t key = i * ncols + c;                  // sorted table: binary search
					uint32_t lo = 0, hi = nfb;
					while(lo < hi) {
						const uint32_t mid = (lo + hi) >> 1;
						if(fb_key[mid] < key) lo = mid + 1; else hi = mid;
					}
					len = 1 + fb_len[lo];
					ft = fb_text + fb_off[lo];
				}
			}
			uint32_t off = len;                                          // inclusive scan of the item lengths
#pragma unroll
			for(int o = 1; o < 32; o <<= 1) {
				const uint32_t t = __shfl_up_sync(0xffffffffu, off, o);
				if(lane >= o)
					off += t;
			}
			const uint32_t tot = __shfl_sync(0xffffffffu, off, 31);
			off -= len;
			if(((a + mis) & 15) + n + tot > TX_BUF) {
				tx_flush(buf, out, a, n, lane);
				a += n;
				n = 0;
			}
			if(((a + mis) & 15) + tot > TX_BUF) {
				// only long host-printed values get here: written straight to the output
				if(len) {
					unsigned char* dst = reinterpret_cast<unsigned char*>(out + a + off);
					tx_put<P>(dst, fast, neg, ip, fp, len, ft);
				}
				a += tot;
				__syncwarp();
				continue;
			}
			if(len)
				tx_put<P>(buf + ((a + mis) & 15) + n + off, fast, neg, ip, fp, len, ft);
			n += tot;
		}
		if(((a + mis) & 15) + n + 1 > TX_BUF) {
			tx_flush(buf, out, a, n, lane);
			a += n;
			n = 0;
		}
		if(lane == 0)
			buf[((a + mis) & 15) + n] = '\n';
		tx_flush(buf, out, a, n + 1, lane);
	}
}

template <int P>
int format_lrn(abw_ctx* ctx, const double* d_values, uint64_t ld, uint32_t col0, uint32_t ncols, const uint64_t* rows, int rows_on_device, uint64_t line0,
               uint64_t nlines, char* d_text, uint64_t cap, uint64_t* nlines_done, uint64_t* nbytes)
{
	// no line is shorter than a one-digit key, ncols times tab + "0." + P digits, and a newline: more lines than this cannot fit
	const uint64_t min_line = 2 + (uint64_t)ncols * (3 + P);
	const uint64_t n = std::min(nlines - line0, cap / min_line + 1);
	DevBuf<uint64_t> d_rows, offs, tot_cut, fb_key, fb_off;
	DevBuf<uint32_t> line_len, fb_count, fb_len;
	DevBuf<TxFallback> fb;
	DevBuf<char> fb_text;
	const uint64_t* r = nullptr;
	if(rows) {
		if(rows_on_device)
			r = rows + line0;
		else {
			ABW_CUDA(ctx, d_rows.alloc(n));
			ABW_CUDA(ctx, cudaMemcpyAsync(d_rows.p, rows + line0, n * sizeof(uint64_t), cudaMemcpyHostToDevice, ctx->stream));
			r = d_rows.p;
		}
	}
	ABW_CUDA(ctx, line_len.alloc(n));
	ABW_CUDA(ctx, offs.alloc(n));
	ABW_CUDA(ctx, tot_cut.alloc(4));
	ABW_CUDA(ctx, fb_count.alloc(1));
	const unsigned int blocks = (unsigned int)std::min<uint64_t>(abw_div_up(n, TX_WARPS), (uint64_t)ctx->sm_count * 16);
	uint32_t fb_cap = (uint32_t)std::min<uint64_t>((uint64_t)n * ncols, 1u << 12), nfb = 0;
	for(;;) {
		ABW_CUDA(ctx, fb.alloc(std::max<uint32_t>(fb_cap, 1)));
		ABW_CUDA(ctx, cudaMemsetAsync(fb_count.p, 0, sizeof(uint32_t), ctx->stream));
		ABW_LAUNCH(ctx, k_lrn_text_len<P>, blocks, TX_WARPS * 32, 0, d_values, ld, col0, ncols, r, line0, n, line_len.p, fb.p, fb_cap, fb_count.p);
		ABW_CUDA(ctx, abw_fetch(ctx, &nfb, fb_count.p, sizeof(uint32_t)));
		ABW_CUDA(ctx, abw_sync(ctx));
		if(nfb <= fb_cap)
			break;
		fb_cap = nfb;                                                   // more values off the integer path than room: once more with room for all
	}
	if(nfb) {
		// the values off the integer path are printed by the C library, as printf would; the table is sorted by (line, column) for the writer
		std::vector<TxFallback> h(nfb);
		ABW_CUDA(ctx, abw_fetch(ctx, h.data(), fb.p, sizeof(TxFallback) * nfb));
		ABW_CUDA(ctx, abw_sync(ctx));
		std::sort(h.begin(), h.end(), [](const TxFallback& x, const TxFallback& y) { return x.key < y.key; });
		std::vector<uint64_t> key(nfb), off(nfb);
		std::vector<uint32_t> len(nfb);
		std::string text;
		char tmp[512];
		for(uint32_t k = 0; k < nfb; k++) {
			const int w = snprintf(tmp, sizeof(tmp), P == 3? "%.3lf" : "%lf", h[k].v);
			key[k] = h[k].key;
			off[k] = text.size();
			len[k] = (uint32_t)w;
			text.append(tmp, (size_t)w);
		}
		ABW_CUDA(ctx, fb_key.alloc(nfb));
		ABW_CUDA(ctx, fb_off.alloc(nfb));
		ABW_CUDA(ctx, fb_len.alloc(nfb));
		ABW_CUDA(ctx, fb_text.alloc(text.size()));
		ABW_CUDA(ctx, cudaMemcpyAsync(fb_key.p, key.data(), nfb * sizeof(uint64_t), cudaMemcpyHostToDevice, ctx->stream));
		ABW_CUDA(ctx, cudaMemcpyAsync(fb_off.p, off.data(), nfb * sizeof(uint64_t), cudaMemcpyHostToDevice, ctx->stream));
		ABW_CUDA(ctx, cudaMemcpyAsync(fb_len.p, len.data(), nfb * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
		ABW_CUDA(ctx, cudaMemcpyAsync(fb_text.p, text.data(), text.size(), cudaMemcpyHostToDevice, ctx->stream));
		ABW_LAUNCH(ctx, k_lrn_text_fb_len, abw_div_up(nfb, 256), 256, 0, fb_key.p, fb_len.p, nfb, ncols, line_len.p);
		ABW_CUDA(ctx, abw_sync(ctx));                                   // the host vectors are locals
	}
	ABW_CHECK(abw_exclusive_scan_u32_to_u64(ctx, line_len.p, offs.p, n, tot_cut.p));
	ABW_LAUNCH(ctx, k_lrn_text_cut, 1, 1, 0, offs.p, tot_cut.p, n, cap, tot_cut.p + 1);
	ABW_LAUNCH(ctx, k_lrn_text_write<P>, blocks, TX_WARPS * 32, 0, d_values, ld, col0, ncols, r, line0, tot_cut.p + 1, offs.p, fb_key.p, fb_off.p, fb_len.p, nfb,
	           fb_text.p, d_text);
	uint64_t h_cut[3] = {0, 0, 0};
	ABW_CUDA(ctx, abw_fetch(ctx, h_cut, tot_cut.p + 1, sizeof(h_cut)));
	ABW_CUDA(ctx, abw_sync(ctx));
	*nlines_done = h_cut[0];
	*nbytes = h_cut[1];
	if(h_cut[0] == 0) {
		*nbytes = h_cut[2];
		return abw_fail(ctx, ABW_ERR_ARG, "abw_format_lrn: the first line does not fit the text buffer (nbytes holds its size)");
	}
	return ABW_OK;
}

}  // namespace

extern "C" int abw_format_lrn(abw_ctx* ctx, const double* d_values, uint64_t ld, uint32_t col0, uint32_t ncols, const uint64_t* rows, int rows_on_device,
                              uint64_t line0, uint64_t nlines, int fmt, char* d_text, uint64_t cap, uint64_t* nlines_done, uint64_t* nbytes)
{
	if(!ctx || !nlines_done || !nbytes || line0 > nlines || (fmt != ABW_TEXT_3LF && fmt != ABW_TEXT_LF) || ncols > TX_MAX_COLS ||
	   (nlines > line0 && (!d_values || !d_text)))
		return abw_fail(ctx, ABW_ERR_ARG, "abw_format_lrn: bad argument");
	ABW_ENTER(ctx);
	*nlines_done = 0;
	*nbytes = 0;
	if(nlines == line0)
		return ABW_OK;
	return fmt == ABW_TEXT_3LF? format_lrn<3>(ctx, d_values, ld, col0, ncols, rows, rows_on_device, line0, nlines, d_text, cap, nlines_done, nbytes)
	                          : format_lrn<6>(ctx, d_values, ld, col0, ncols, rows, rows_on_device, line0, nlines, d_text, cap, nlines_done, nbytes);
}
