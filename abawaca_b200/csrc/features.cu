// Feature stage of abawaca-build on the device: 2-bit packing, windowing, k-mer signatures, coverage.
//
// Data layout in HBM (abw_seqset): every scaffold starts at a base offset that is a multiple of 128, so that
//   packed : 2 bits/base, 16 bases per u32, base i of the scaffold at bits [2*(i%16), +2) of word base/16+i/16
//            (A=0 C=1 G=2 T=3; non-ACGT positions hold 0),
//   valid  : 1 bit/base, set for A/C/G/T (after upper-casing),
//   nmask  : 1 bit/base, set for the literal 'N' only (quirk Q2: IUPAC codes are bases for windowing, but break k-mers)
// are all 16-byte aligned per scaffold and can be fetched with 128-bit loads.
#include "common.cuh"
#include <algorithm>

#include "features.cuh"

namespace {

// ---------------------------------------------------------------------------------------------------
// pack
// ---------------------------------------------------------------------------------------------------
// bit 7 of every byte of x that equals the corresponding byte of c4 (exact: the classic zero-byte test on x ^ c4)
__device__ __forceinline__ uint32_t eq_bytes(uint32_t x, uint32_t c4)
{
	const uint32_t y = x ^ c4;
	const uint32_t t = (y & 0x7F7F7F7Fu) + 0x7F7F7F7Fu;
	return ~(t | y) & 0x80808080u;
}

// 4 ASCII characters -> 8 bits of 2-bit codes + 4 valid bits + 4 N bits (+ GC count, + lower-case-n flag), in plain integer arithmetic (the SIMD-in-a-word
// compare intrinsics are emulated on this architecture and made the kernel instruction bound).  Clearing bit 5 maps a-z onto A-Z (toupper() for letters,
// String.cpp:44) and maps no other byte onto one of A C G T N; A|C and C|G differ in one bit each, so four byte-wise equality tests decide everything.
__device__ __forceinline__ void classify4(uint32_t w, uint32_t& code8, uint32_t& valid4, uint32_t& n4, uint32_t& gc, uint32_t& bad)
{
	const uint32_t u = w & 0xDFDFDFDFu;
	const uint32_t eAC = eq_bytes(u & 0xFDFDFDFDu, 0x41414141u);          // A (0x41) or C (0x43)
	const uint32_t eCG = eq_bytes(u & 0xFBFBFBFBu, 0x43434343u);          // C (0x43) or G (0x47)
	const uint32_t eT = eq_bytes(u, 0x54545454u), eN = eq_bytes(u, 0x4E4E4E4Eu);
	bad |= eN & (w << 2);                                   // bit 5 set: 'n' throws in the reference (String.cpp:47-49)
	const uint32_t lo = (eAC & eCG) | eT, hi = (eCG & ~eAC) | eT;         // A=0 C=1 G=2 T=3
	const uint32_t x = (lo >> 7) | (hi >> 6);               // one 2-bit code per byte, 0 for every other character
	code8 = (x * 0x01041040u) >> 24;                        // the four 2-bit fields side by side (the partial products do not overlap)
	valid4 = (((eAC | eCG | eT) >> 7) * 0x01020408u) >> 24; // bit 0 of each byte -> 4 bits
	n4 = ((eN >> 7) * 0x01020408u) >> 24;
	gc += __popc(eCG);
}

// One warp per scaffold; per step a lane takes 16 consecutive bases (one 16-byte window of the text, read as two aligned 16-byte loads and shifted into
// place -- the offset of a scaffold in the text is arbitrary, its place in the packed arrays is aligned), i.e. one packed word; a warp step is 512 bases
// with fully coalesced loads and stores, two steps are in flight.  Lane pairs combine their 16 validity / N bits into one word.
__device__ __forceinline__ void pack16(const unsigned char* __restrict__ ascii, uint64_t ascii_bytes, uint64_t a, uint32_t cnt, uint32_t& code, uint32_t& v16, uint32_t& n16,
                                       uint32_t& nGC, uint32_t& bad)
{
	uint32_t w[4];
	const uint64_t al = a & ~15ull;
	if(cnt == 16 && al + 32 <= ascii_bytes) {
		const uint4 A = __ldg(reinterpret_cast<const uint4*>(ascii + al)), B = __ldg(reinterpret_cast<const uint4*>(ascii + al + 16));
		const uint32_t sh = (uint32_t)(a & 15), r8 = (sh & 3u) * 8u;
		switch(sh >> 2) {                                   // uniform over the warp: every lane of a scaffold has the same misalignment
		case 0: w[0] = __funnelshift_r(A.x, A.y, r8); w[1] = __funnelshift_r(A.y, A.z, r8); w[2] = __funnelshift_r(A.z, A.w, r8); w[3] = __funnelshift_r(A.w, B.x, r8); break;
		case 1: w[0] = __funnelshift_r(A.y, A.z, r8); w[1] = __funnelshift_r(A.z, A.w, r8); w[2] = __funnelshift_r(A.w, B.x, r8); w[3] = __funnelshift_r(B.x, B.y, r8); break;
		case 2: w[0] = __funnelshift_r(A.z, A.w, r8); w[1] = __funnelshift_r(A.w, B.x, r8); w[2] = __funnelshift_r(B.x, B.y, r8); w[3] = __funnelshift_r(B.y, B.z, r8); break;
		default: w[0] = __funnelshift_r(A.w, B.x, r8); w[1] = __funnelshift_r(B.x, B.y, r8); w[2] = __funnelshift_r(B.y, B.z, r8); w[3] = __funnelshift_r(B.z, B.w, r8); break;
		}
	}
	else {
#pragma unroll
		for(int i = 0; i < 4; i++) {
			uint32_t x = 0;
#pragma unroll
			for(int j = 0; j < 4; j++) {
				const uint32_t k = i * 4 + j;
				const uint32_t c = (k < cnt)? (uint32_t)ascii[a + k] : 0u;
				x |= c << (8 * j);
			}
			w[i] = x;
		}
	}
	code = 0; v16 = 0; n16 = 0;
#pragma unroll
	for(int i = 0; i < 4; i++) {
		uint32_t c8, v4, n4;
		classify4(w[i], c8, v4, n4, nGC, bad);
		code |= c8 << (8 * i);
		v16 |= v4 << (4 * i);
		n16 |= n4 << (4 * i);
	}
}

__global__ void __launch_bounds__(256) k_pack(const unsigned char* __restrict__ ascii, uint64_t ascii_bytes, const uint64_t* __restrict__ offsets,
                                              const uint64_t* __restrict__ base, uint32_t nscaf, uint32_t* __restrict__ packed, uint32_t* __restrict__ valid,
                                              uint32_t* __restrict__ nmask, unsigned long long* __restrict__ countN, unsigned long long* __restrict__ countGC,
                                              int* __restrict__ err)
{
	abw_grid_wait();
	const int lane = threadIdx.x & 31;
	const uint64_t warp0 = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
	for(uint64_t s = warp0; s < nscaf; s += nwarps) {
		const uint64_t off = offsets[s], len = offsets[s + 1] - off, b0 = base[s], padded = base[s + 1] - b0;     // padded: a multiple of 128 bases
		uint32_t nN = 0, nGC = 0, bad = 0;
		for(uint64_t p0 = 0; p0 < padded; p0 += 1024) {
			uint32_t code[2], v16[2], n16[2];
#pragma unroll
			for(int h = 0; h < 2; h++) {
				const uint64_t p = p0 + 512 * h + 16 * lane;     // first base of this lane's piece within the scaffold
				code[h] = 0; v16[h] = 0; n16[h] = 0;
				if(p < len)
					pack16(ascii, ascii_bytes, off + p, (uint32_t)min((uint64_t)16, len - p), code[h], v16[h], n16[h], nGC, bad);
			}
#pragma unroll
			for(int h = 0; h < 2; h++) {
				const uint64_t p = p0 + 512 * h + 16 * lane;
				// the neighbour's 16 bits complete the word of 32 positions (every lane takes part in the exchange)
				const uint32_t v = v16[h] | (__shfl_down_sync(0xffffffffu, v16[h], 1) << 16), nm = n16[h] | (__shfl_down_sync(0xffffffffu, n16[h], 1) << 16);
				nN += __popc(n16[h]);
				if(p < padded) {
					packed[(b0 + p) >> 4] = code[h];
					if((lane & 1) == 0) {
						valid[(b0 + p) >> 5] = v;
						nmask[(b0 + p) >> 5] = nm;
					}
				}
			}
		}
#pragma unroll
		for(int o = 16; o > 0; o >>= 1) {
			nN += __shfl_xor_sync(0xffffffffu, nN, o);
			nGC += __shfl_xor_sync(0xffffffffu, nGC, o);
			bad |= __shfl_xor_sync(0xffffffffu, bad, o);
		}
		if(lane == 0) {
			countN[s] = nN;
			countGC[s] = nGC;
			if(bad)
				atomicExch(err, 1);
		}
	}
}

// ---------------------------------------------------------------------------------------------------
// windowing, abawaca-build.cpp:198-228
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ void window_plan(uint64_t len, uint64_t nN, uint64_t window, uint64_t& nbps, uint64_t& count)
{
	uint64_t nonN = len - nN;
	uint64_t nsegments = nonN / window;                     // :202
	if(nsegments == 0)
		nsegments = 1;                                      // :204-205
	nbps = nonN / nsegments;                                // :206
	// a window closes every time nbps non-N characters were seen (:210-224); with no non-N base at all the
	// test `nbps_segment == nbps` is 0 == 0 at every character, so every character becomes a window
	count = (nbps > 0)? nonN / nbps : len;
}


__global__ void k_seg_count(const uint64_t* __restrict__ len, const unsigned long long* __restrict__ countN, uint32_t nscaf, uint64_t window, uint64_t* __restrict__ counts)
{
	abw_grid_wait();
	uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
	if(s < nscaf) {
		uint64_t nbps, count;
		window_plan(len[s], countN[s], window, nbps, count);
		counts[s] = count;
	}
}

// one warp per scaffold walks the N mask; window j ends at the (j*nbps)-th non-N character
__global__ void __launch_bounds__(256) k_seg_fill(const uint64_t* __restrict__ len, const unsigned long long* __restrict__ countN, const uint64_t* __restrict__ base,
                                                  const uint32_t* __restrict__ nmask, uint32_t nscaf, uint64_t window, const uint64_t* __restrict__ seg_first,
                                                  uint32_t* __restrict__ seg_scaf, uint64_t* __restrict__ seg_start, uint64_t* __restrict__ seg_end,
                                                  uint64_t* __restrict__ seg_nonN, uint64_t* __restrict__ seg_gbase, uint4* __restrict__ scaf_info)
{
	abw_grid_wait();
	const int lane = threadIdx.x & 31;
	const uint64_t warp0 = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
	for(uint64_t s = warp0; s < nscaf; s += nwarps) {
		const uint64_t L = len[s], b0 = base[s], first = seg_first[s];
		uint64_t nbps, count;
		window_plan(L, countN[s], window, nbps, count);
		if(lane == 0)
			{
			// .w: bits 32.. of nbps (coverage then searches instead of guessing), or COV_REGULAR for a scaffold without N whose windows
			// are exactly [j nbps + 1, (j + 1) nbps]: coverage then needs no window table at all
			uint32_t hi = (uint32_t)min(nbps >> 32, (uint64_t)0x7FFFFFFFu);
			if(countN[s] == 0 && nbps > 0 && hi == 0)
				hi = COV_REGULAR;
			scaf_info[s] = make_uint4((uint32_t)first, (uint32_t)min(count, (uint64_t)0xFFFFFFFFu), (uint32_t)nbps, hi);
		}
		if(count == 0)
			continue;
		if(nbps == 0) {
			for(uint64_t i = lane; i < count; i += 32) {
				seg_scaf[first + i] = (uint32_t)s;
				seg_start[first + i] = i + 1;
				seg_end[first + i] = i + 1;
				seg_nonN[first + i] = 0;
				seg_gbase[first + i] = b0 + i;
			}
			continue;
		}
		if(lane == 0) {
			seg_start[first] = 1;
			seg_gbase[first] = b0;
		}
		for(uint64_t i = lane; i < count; i += 32) {
			seg_scaf[first + i] = (uint32_t)s;
			seg_nonN[first + i] = nbps;
		}
		const uint64_t units = (L + 31) >> 5;
		uint64_t carry = 0;
		for(uint64_t u0 = 0; u0 < units; u0 += 32) {
			uint64_t u = u0 + lane;
			uint32_t bits = 0;
			if(u < units) {
				uint32_t in_range = (L - (u << 5) >= 32)? 0xFFFFFFFFu : ((1u << (uint32_t)(L - (u << 5))) - 1u);
				bits = ~nmask[(b0 >> 5) + u] & in_range;
			}
			uint32_t c = __popc(bits), incl = c;
#pragma unroll
			for(int o = 1; o < 32; o <<= 1) {
				uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
				if(lane >= o)
					incl += t;
			}
			uint64_t before = carry + incl - c, after = carry + incl;
			for(uint64_t j = before / nbps + 1; j * nbps <= after && j <= count; j++) {
				uint32_t k = (uint32_t)(j * nbps - before);          // the k-th set bit of this word closes window j
				uint32_t bit = __fns(bits, 0, k);
				uint64_t pos1 = (u << 5) + bit + 1;                   // 1-based, :216
				seg_end[first + j - 1] = pos1;
				if(j < count) {
					seg_start[first + j] = pos1 + 1;                  // :221-222
					seg_gbase[first + j] = b0 + pos1;
				}
			}
			carry += __shfl_sync(0xffffffffu, incl, 31);
		}
	}
}

// ---------------------------------------------------------------------------------------------------
// k-mer signature, abawaca-build.cpp:103-174
// ---------------------------------------------------------------------------------------------------
// dimension tables: for each of the 180 canonical dims the k, and the two little-endian codes (mer, reverse complement)
// Kept in GLOBAL memory and copied to shared memory by every CTA: lanes index them with different addresses, which the
// indexed-constant path serialises (round 1 ncu: ADU pipe 72 % busy with these lookups when they were __constant__).
__device__ uint32_t g_dim_tab[ABW_NKMER_DIMS];              // k | code_a << 8 | code_b << 16
__device__ double   g_milli[1001];                          // m / 1000.0

constexpr int KM_WARPS = 8;
constexpr int KM_GROUPS = 4;                                // sub-histograms per warp: lanes 8g..8g+7 share one

// Per warp.  hist is bin-major and interleaved by group: word = bin * 4 + group, so two lanes can only hit the same bank when they are in the
// same group of eight (micro-benchmark scripts/ubench_hist.cu on B200, updates per clock and SM: 13.3 in this layout with fire-and-forget
// shared atomics, 14.0 with eight groups at twice the footprint, 8.6 for a private byte histogram per lane updated with load/add/store,
// 10.4 for 16-bit counters or for 5-mer bins counted at every second position).  5.4 KB per warp: five CTAs of eight warps per SM.
struct __align__(16) KmWarpSmem {
	uint32_t hist[256 * KM_GROUPS];
	uint32_t cnt4[256];
	uint32_t cnt3[64];
	uint32_t cnt2[16];
	uint32_t cnt1[4];
	uint32_t tot[4];
	float    inv_tot[4];            // 1 / total_k, only used to form an integer quotient that is then verified exactly
	uint32_t pad[4];
};

// A warp per window; lane l takes the 16-base words l, l+32, ... of the window straight from global memory (the packed stream and the
// validity bits of neighbouring words share cache lines).  A word whose 16 four-mers are all valid costs 16 shared atomics; the first and
// last words of the window and words next to a non-ACGT character go through the per-position path.
template <int KIND>
__global__ void __launch_bounds__(KM_WARPS * 32) k_kmer(const uint32_t* __restrict__ packed, const uint32_t* __restrict__ valid, const uint64_t* __restrict__ seg_gbase,
                                                        const uint64_t* __restrict__ seg_start, const uint64_t* __restrict__ seg_end, uint64_t nseg, int skip_A,
                                                        double* __restrict__ rows, uint64_t ld, uint32_t col0)
{
	abw_grid_wait();
	__shared__ uint32_t sm_dim_tab[ABW_NKMER_DIMS];
	__shared__ KmWarpSmem sm_warp[KM_WARPS];
	KmWarpSmem* sm = sm_warp + (threadIdx.x >> 5);
	const int lane = threadIdx.x & 31;
	for(int i = threadIdx.x; i < ABW_NKMER_DIMS; i += blockDim.x)
		sm_dim_tab[i] = g_dim_tab[i];
	for(int i = lane; i < 256 * KM_GROUPS; i += 32)
		sm->hist[i] = 0;
	__syncthreads();
	uint32_t* const myhist = sm->hist + (lane >> 3);        // + bin * KM_GROUPS
	const uint64_t warp0 = (uint64_t)blockIdx.x * KM_WARPS + (threadIdx.x >> 5), nwarps = (uint64_t)gridDim.x * KM_WARPS;
	for(uint64_t g = warp0; g < nseg; g += nwarps) {
		const uint64_t gb = seg_gbase[g];
		const uint64_t pos_end = gb + (seg_end[g] - seg_start[g] + 1);
		for(int i = lane; i < 64 + 16 + 4 + 4; i += 32)
			sm->cnt3[i] = 0;                                // cnt3, cnt2, cnt1, tot are contiguous: these receive the run-end windows
		__syncwarp();
		const uint64_t wend = (pos_end + 15) >> 4;
		for(uint64_t wa = (gb >> 4) + lane; wa < wend; wa += 32) {
			const uint32_t w_lo = __ldg(packed + wa), w_hi = __ldg(packed + wa + 1);
			const uint32_t va = __ldg(valid + (wa >> 1)), vb = __ldg(valid + (wa >> 1) + 1);
			uint32_t v = __funnelshift_r(va, vb, (uint32_t)(wa & 1) * 16) & 0x7FFFFu;       // 16 positions + 3 lookahead
			const uint64_t p0 = wa << 4;
			// positions outside [gb, pos_end) never hold a base of this window
			if(p0 < gb)
				v &= 0xFFFFFFFFu << (uint32_t)(gb - p0);
			if(pos_end - p0 < 19)
				v &= (1u << (uint32_t)(pos_end - p0)) - 1u;
			const uint32_t v1 = v & 0xFFFFu, v2 = v1 & (v >> 1), v3 = v2 & (v >> 2), v4 = v3 & (v >> 3);
			// s[i] = the window shifted by i bases: 4-mer t = 4 j + i is byte j of s[i]
			uint32_t sh[4];
			sh[0] = w_lo;
			sh[1] = __funnelshift_r(w_lo, w_hi, 2);
			sh[2] = __funnelshift_r(w_lo, w_hi, 4);
			sh[3] = __funnelshift_r(w_lo, w_hi, 6);
			if(v4 == 0xFFFFu) {
#pragma unroll
				for(int i = 0; i < 4; i++) {
#pragma unroll
					for(int j = 0; j < 4; j++)
						atomicAdd(myhist + ((sh[i] >> (8 * j)) & 0xFFu) * KM_GROUPS, 1u);
				}
			}
			else if(v1) {
				// windows broken by a non-ACGT character or by the end of the segment (:131,147 key = 0)
				const uint32_t e3 = v3 & ~v4, e2 = v2 & ~v3, e1 = v1 & ~v2;
#pragma unroll
				for(int i = 0; i < 4; i++) {
#pragma unroll
					for(int j = 0; j < 4; j++) {
						const int t = 4 * j + i;
						const uint32_t x = (sh[i] >> (8 * j)) & 0xFFu;
						if((v4 >> t) & 1u)
							atomicAdd(myhist + x * KM_GROUPS, 1u);
						else if((e3 >> t) & 1u)
							atomicAdd(&sm->cnt3[x & 63u], 1u);
						else if((e2 >> t) & 1u)
							atomicAdd(&sm->cnt2[x & 15u], 1u);
						else if((e1 >> t) & 1u)
							atomicAdd(&sm->cnt1[x & 3u], 1u);
					}
				}
			}
		}
		__syncwarp();
		// fold the sub-histograms: lane l owns bins l, l+32, ..., l+224 (four consecutive words each) and clears them
		{
			uint32_t t4 = 0;
#pragma unroll
			for(int j = 0; j < 8; j++) {
				const int bin = lane + 32 * j;
				uint4* hp = reinterpret_cast<uint4*>(sm->hist + bin * KM_GROUPS);
				const uint4 a = hp[0];
				hp[0] = make_uint4(0, 0, 0, 0);
				const uint32_t c = a.x + a.y + a.z + a.w;
				sm->cnt4[bin] = c;
				t4 += c;
			}
			t4 = __reduce_add_sync(0xffffffffu, t4);
			__syncwarp();
			// lower orders: every valid 4-mer start is a valid 3-mer start, etc.; cnt3/cnt2/cnt1 hold the run-end extras
			uint32_t a = sm->cnt4[lane] + sm->cnt4[lane + 64] + sm->cnt4[lane + 128] + sm->cnt4[lane + 192];
			uint32_t b = sm->cnt4[lane + 32] + sm->cnt4[lane + 96] + sm->cnt4[lane + 160] + sm->cnt4[lane + 224];
			a += sm->cnt3[lane];
			b += sm->cnt3[lane + 32];
			sm->cnt3[lane] = a;
			sm->cnt3[lane + 32] = b;
			const uint32_t t3 = __reduce_add_sync(0xffffffffu, a + b);
			__syncwarp();
			uint32_t c2 = 0;
			if(lane < 16) {
				c2 = sm->cnt2[lane] + sm->cnt3[lane] + sm->cnt3[lane + 16] + sm->cnt3[lane + 32] + sm->cnt3[lane + 48];
				sm->cnt2[lane] = c2;
			}
			const uint32_t t2 = __reduce_add_sync(0xffffffffu, c2);
			__syncwarp();
			uint32_t c1 = 0;
			if(lane < 4) {
				c1 = sm->cnt1[lane] + sm->cnt2[lane] + sm->cnt2[lane + 4] + sm->cnt2[lane + 8] + sm->cnt2[lane + 12];
				sm->cnt1[lane] = c1;
			}
			const uint32_t t1 = __reduce_add_sync(0xffffffffu, c1);
			if(lane < 4) {
				const uint32_t tk = (lane == 0)? t1 : (lane == 1)? t2 : (lane == 2)? t3 : t4;
				sm->tot[lane] = tk;
				sm->inv_tot[lane] = tk? 1.0f / (float)tk : 0.0f;
			}
			__syncwarp();
		}
		// 180 canonical dimensions: dims[canon] += count/total for the mer and for its reverse complement (:171)
		for(int d = lane; d < ABW_NKMER_DIMS; d += 32) {
			const uint32_t ent = sm_dim_tab[d];
			const int k = ent & 0xFFu;
			const uint32_t* cnt = (k == 4)? sm->cnt4 : (k == 3)? sm->cnt3 : (k == 2)? sm->cnt2 : sm->cnt1;
			const uint32_t ca = (ent >> 8) & 0xFFu, cb = (ent >> 16) & 0xFFu;
			const uint32_t c1 = cnt[ca], c2 = (cb != ca)? cnt[cb] : 0u;
			const uint32_t t = sm->tot[k - 1];
			double out = 0.0;
			if(t != 0 && (c1 + c2) != 0) {
				bool exact_path = (KIND != ABW_FEAT_TRUNC3) || (c1 + c2) > 4000000u || t > (1u << 28);
				if(!exact_path) {
					// int(1000*(c1/t + c2/t)) equals floor(1000*(c1+c2)/t) whenever the quotient is not an integer: the rounding
					// error of the three fp64 operations (< 1e-12) is far below the distance 1/t to the next integer.  The quotient
					// (at most 1000) is formed in single precision, off by at most one, and verified exactly in integers.
					const uint32_t num = 1000u * (c1 + c2);
					uint32_t m = (uint32_t)__float2uint_rz((float)num * sm->inv_tot[k - 1]);
					int32_t r = (int32_t)(num - m * t);
					if(r < 0) { m--; r += (int32_t)t; }
					else if((uint32_t)r >= t) { m++; r -= (int32_t)t; }
					if(r != 0)
						out = g_milli[m];
					else
						exact_path = true;
				}
				if(exact_path) {
					double x = (c1? __ddiv_rn((double)c1, (double)(int)t) : 0.0);
					if(c2)
						x = __dadd_rn(x, __ddiv_rn((double)c2, (double)(int)t));
					out = (KIND == ABW_FEAT_TRUNC3)? __ddiv_rn((double)__double2int_rz(__dmul_rn(1000.0, x)), 1000.0) : x;
				}
			}
			if(!(skip_A && d == 0))
				rows[g * ld + col0 + d - (skip_A? 1 : 0)] = out;
		}
		__syncwarp();
	}
}

// integer thousandths of the columns [col0, col0 + ncols) of a row-major matrix (abw_rows_to_milli)
template <typename OutT>
__global__ void __launch_bounds__(256) k_rows_milli(const double* __restrict__ rows, uint64_t nrows, uint64_t ld, uint32_t col0, uint32_t ncols, OutT* __restrict__ out,
                                                    int* __restrict__ inexact)
{
	abw_grid_wait();
	const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
	bool bad = false;
	if(i < nrows * ncols) {
		const uint64_t r = i / ncols;
		const uint32_t c = (uint32_t)(i - r * ncols);
		const double v = rows[r * ld + col0 + c];
		const double k = rint(__dmul_rn(v, 1000.0));
		const double kmax = (sizeof(OutT) == 2)? 65535.0 : 4294967295.0;
		const bool ok = (k >= 0.0) && (k <= kmax) && (__ddiv_rn(k, 1000.0) == v) && !(v == 0.0 && signbit(v));
		out[i] = ok? (OutT)(unsigned long long)k : (OutT)0;
		bad = !ok;
	}
	const uint32_t nb = __popc(__ballot_sync(0xffffffffu, bad));
	if(nb && (threadIdx.x & 31) == 0)
		atomicAdd(inexact, (int)nb);
}

bool g_tables_ready[64] = {};

int upload_tables(abw_ctx* ctx)
{
	if(ctx->device >= 0 && ctx->device < 64 && g_tables_ready[ctx->device])
		return ABW_OK;
	uint8_t dk[ABW_NKMER_DIMS];
	uint16_t da[ABW_NKMER_DIMS], db[ABW_NKMER_DIMS];
	int next = 0;
	int dim_of[5][256];
	for(int k = 1; k <= 4; k++) {
		int n = 1 << (2 * k);
		for(int code = 0; code < n; code++) {              // big-endian code = lexicographic order, abawaca-build.cpp:90-99
			int rc = 0, c = code;
			for(int i = 0; i < k; i++) { rc = (rc << 2) | (3 - (c & 3)); c >>= 2; }
			auto to_le = [k](int be) { int le = 0; for(int i = 0; i < k; i++) { le |= ((be >> (2 * (k - 1 - i))) & 3) << (2 * i); } return le; };
			if(rc < code)
				dim_of[k][code] = dim_of[k][rc];
			else {
				dim_of[k][code] = next;
				dk[next] = (uint8_t)k;
				da[next] = (uint16_t)to_le(code);
				db[next] = (uint16_t)to_le(rc);
				next++;
			}
		}
	}
	if(next != ABW_NKMER_DIMS)
		return abw_fail(ctx, ABW_ERR_ARG, "internal: canonical k-mer table size");
	double milli[1001];
	for(int m = 0; m <= 1000; m++)
		milli[m] = (double)m / 1000.0;
	uint32_t tab[ABW_NKMER_DIMS];
	for(int i = 0; i < ABW_NKMER_DIMS; i++)
		tab[i] = (uint32_t)dk[i] | ((uint32_t)da[i] << 8) | ((uint32_t)db[i] << 16);
	ABW_CUDA(ctx, cudaMemcpyToSymbol(g_dim_tab, tab, sizeof(tab)));
	ABW_CUDA(ctx, cudaMemcpyToSymbol(g_milli, milli, sizeof(milli)));
	if(ctx->device >= 0 && ctx->device < 64)
		g_tables_ready[ctx->device] = true;
	return ABW_OK;
}

}  // namespace

// ===================================================================================================
// C ABI
// ===================================================================================================
extern "C" {

static int pack_impl(abw_ctx* ctx, abw_seqset* s, const char* ascii, int ascii_on_device, const uint64_t* h_offsets, uint32_t nscaf)
{
	s->nscaf = nscaf;
	s->h_len.resize(nscaf);
	s->h_base.resize((size_t)nscaf + 1);
	uint64_t b = 0;
	for(uint32_t i = 0; i < nscaf; i++) {
		if(h_offsets[i + 1] < h_offsets[i])
			return abw_fail(ctx, ABW_ERR_ARG, "abw_pack_sequences: offsets must be non-decreasing");
		s->h_len[i] = h_offsets[i + 1] - h_offsets[i];
		s->h_base[i] = b;
		b += (s->h_len[i] + 127) & ~127ull;
	}
	s->h_base[nscaf] = b;
	s->total_padded = b;
	const uint64_t bytes = h_offsets[nscaf];
	DevBuf<unsigned char> d_ascii;
	DevBuf<uint64_t> d_off;
	DevBuf<int> d_err;
	const unsigned char* src = (const unsigned char*)ascii;
	uint64_t readable = bytes;
	if(!ascii_on_device) {
		ABW_CUDA(ctx, d_ascii.alloc(bytes + 64));
		ABW_CUDA(ctx, cudaMemcpyAsync(d_ascii.p, ascii, bytes, cudaMemcpyHostToDevice, ctx->stream));
		src = d_ascii.p;
		readable = bytes + 64;
	}
	ABW_CUDA(ctx, d_off.alloc((size_t)nscaf + 1));
	ABW_CUDA(ctx, abw_upload_small(ctx, d_off.p, h_offsets, sizeof(uint64_t) * ((size_t)nscaf + 1)));
	ABW_CUDA(ctx, s->len.alloc(nscaf));
	ABW_CUDA(ctx, s->base.alloc((size_t)nscaf + 1));
	ABW_CUDA(ctx, abw_upload_small(ctx, s->len.p, s->h_len.data(), sizeof(uint64_t) * nscaf));
	ABW_CUDA(ctx, abw_upload_small(ctx, s->base.p, s->h_base.data(), sizeof(uint64_t) * ((size_t)nscaf + 1)));
	// + slack so that the k-mer kernel may read one word past a segment
	ABW_CUDA(ctx, s->packed.alloc(b / 16 + 16));
	ABW_CUDA(ctx, s->valid.alloc(b / 32 + 16));
	ABW_CUDA(ctx, s->nmask.alloc(b / 32 + 16));
	ABW_CUDA(ctx, cudaMemsetAsync(s->packed.p + b / 16, 0, 16 * sizeof(uint32_t), ctx->stream));
	ABW_CUDA(ctx, cudaMemsetAsync(s->valid.p + b / 32, 0, 16 * sizeof(uint32_t), ctx->stream));
	ABW_CUDA(ctx, cudaMemsetAsync(s->nmask.p + b / 32, 0, 16 * sizeof(uint32_t), ctx->stream));
	ABW_CUDA(ctx, s->countN.alloc(nscaf));
	ABW_CUDA(ctx, s->countGC.alloc(nscaf));
	ABW_CUDA(ctx, d_err.alloc(1));
	ABW_CUDA(ctx, cudaMemsetAsync(d_err.p, 0, sizeof(int), ctx->stream));
	if(nscaf > 0) {
		unsigned int blocks = (unsigned int)std::min<uint64_t>(abw_div_up((uint64_t)nscaf * 32, 256), (uint64_t)ctx->sm_count * 16);
		ABW_LAUNCH(ctx, k_pack, blocks, 256, 0, src, readable, d_off.p, s->base.p, nscaf, s->packed.p, s->valid.p, s->nmask.p, s->countN.p, s->countGC.p, d_err.p);
	}
	int h_err = 0;
	ABW_CUDA(ctx, abw_fetch(ctx, &h_err, d_err.p, sizeof(int)));
	ABW_CUDA(ctx, abw_sync(ctx));
	if(h_err)
		return abw_fail(ctx, ABW_ERR_ILLEGAL_DNA, "Illegal_DNAString: lower-case 'n' in a sequence (String.cpp:47-49)");
	return ABW_OK;
}

int abw_pack_sequences(abw_ctx* ctx, const char* ascii, int ascii_on_device, const uint64_t* h_offsets, uint32_t nscaf, abw_seqset** out)
{
	if(!ctx || !out || !h_offsets || (!ascii && nscaf && h_offsets[nscaf] > 0))
		return abw_fail(ctx, ABW_ERR_ARG, "abw_pack_sequences: null argument");
	ABW_ENTER(ctx);
	abw_seqset* s = new abw_seqset();
	int rc = pack_impl(ctx, s, ascii, ascii_on_device, h_offsets, nscaf);
	if(rc != ABW_OK) {
		delete s;
		return rc;
	}
	*out = s;
	return ABW_OK;
}

void abw_seqset_destroy(abw_seqset* s) { delete s; }

int abw_seqset_stats(abw_ctx* ctx, const abw_seqset* s, uint64_t* h_count_N, uint64_t* h_count_GC)
{
	if(!ctx || !s)
		return abw_fail(ctx, ABW_ERR_ARG, "abw_seqset_stats: null argument");
	if(h_count_N)
		ABW_CUDA(ctx, abw_fetch(ctx, h_count_N, s->countN.p, sizeof(uint64_t) * s->nscaf));
	if(h_count_GC)
		ABW_CUDA(ctx, abw_fetch(ctx, h_count_GC, s->countGC.p, sizeof(uint64_t) * s->nscaf));
	ABW_CUDA(ctx, abw_sync(ctx));
	return ABW_OK;
}

int abw_segment(abw_ctx* ctx, const abw_seqset* s, uint32_t window_size, abw_segments** out)
{
	if(!ctx || !s || !out || window_size == 0)
		return abw_fail(ctx, ABW_ERR_ARG, "abw_segment: bad argument");
	ABW_ENTER(ctx);
	abw_segments* g = new abw_segments();
	g->nscaf = s->nscaf;
	int rc = [&]() -> int {
		ABW_CUDA(ctx, g->seg_first.alloc((size_t)s->nscaf + 1));
		DevBuf<uint64_t> counts, total;
		ABW_CUDA(ctx, counts.alloc(s->nscaf));
		ABW_CUDA(ctx, total.alloc(1));
		if(s->nscaf > 0)
			ABW_LAUNCH(ctx, k_seg_count, abw_div_up(s->nscaf, 256), 256, 0, s->len.p, s->countN.p, s->nscaf, (uint64_t)window_size, counts.p);
		ABW_CHECK(abw_exclusive_scan_u64(ctx, counts.p, g->seg_first.p, s->nscaf, total.p));
		ABW_CUDA(ctx, abw_fetch(ctx, &g->nseg, total.p, sizeof(uint64_t)));
		ABW_CUDA(ctx, abw_sync(ctx));
		ABW_CUDA(ctx, abw_upload_small(ctx, g->seg_first.p + s->nscaf, &g->nseg, sizeof(uint64_t)));
		ABW_CUDA(ctx, g->seg_scaf.alloc(g->nseg));
		ABW_CUDA(ctx, g->seg_start.alloc(g->nseg));
		ABW_CUDA(ctx, g->seg_end.alloc(g->nseg));
		ABW_CUDA(ctx, g->seg_nonN.alloc(g->nseg));
		ABW_CUDA(ctx, g->seg_gbase.alloc(g->nseg));
		ABW_CUDA(ctx, g->scaf_info.alloc(s->nscaf));
		ABW_CUDA(ctx, cudaMemsetAsync(g->scaf_info.p, 0, sizeof(uint4) * s->nscaf, ctx->stream));
		if(s->nscaf > 0 && g->nseg > 0) {
			unsigned int blocks = (unsigned int)std::min<uint64_t>(abw_div_up((uint64_t)s->nscaf * 32, 256), (uint64_t)ctx->sm_count * 16);
			ABW_LAUNCH(ctx, k_seg_fill, blocks, 256, 0, s->len.p, s->countN.p, s->base.p, s->nmask.p, s->nscaf, (uint64_t)window_size, g->seg_first.p,
			           g->seg_scaf.p, g->seg_start.p, g->seg_end.p, g->seg_nonN.p, g->seg_gbase.p, g->scaf_info.p);
		}
		ABW_CUDA(ctx, abw_sync(ctx));
		return ABW_OK;
	}();
	if(rc != ABW_OK) {
		delete g;
		return rc;
	}
	*out = g;
	return ABW_OK;
}

void abw_segments_destroy(abw_segments* g) { delete g; }

int abw_rows_to_milli(abw_ctx* ctx, const double* d_rows, uint64_t nrows, uint64_t ld, uint32_t col0, uint32_t ncols, int bits, void* d_out, int32_t* d_inexact)
{
	if(!ctx || !d_rows || !d_out || !d_inexact || (bits != 16 && bits != 32))
		return abw_fail(ctx, ABW_ERR_ARG, "abw_rows_to_milli: bad argument");
	if(ld < (uint64_t)col0 + ncols)
		return abw_fail(ctx, ABW_ERR_ARG, "abw_rows_to_milli: row stride too small");
	ABW_ENTER(ctx);
	if(nrows == 0 || ncols == 0)
		return ABW_OK;
	const unsigned int blocks = abw_div_up(nrows * ncols, 256);
	if(bits == 16)
		ABW_LAUNCH(ctx, k_rows_milli<uint16_t>, blocks, 256, 0, d_rows, nrows, ld, col0, ncols, (uint16_t*)d_out, (int*)d_inexact);
	else
		ABW_LAUNCH(ctx, k_rows_milli<uint32_t>, blocks, 256, 0, d_rows, nrows, ld, col0, ncols, (uint32_t*)d_out, (int*)d_inexact);
	return ABW_OK;
}

uint64_t abw_segments_count(const abw_segments* g) { return g? g->nseg : 0; }

int abw_segments_get(abw_ctx* ctx, const abw_segments* g, uint64_t* h_seg_first, uint32_t* h_seg_scaf, uint64_t* h_seg_start, uint64_t* h_seg_end, uint64_t* h_seg_nonN)
{
	if(!ctx || !g)
		return abw_fail(ctx, ABW_ERR_ARG, "abw_segments_get: null argument");
	if(h_seg_first)
		ABW_CUDA(ctx, abw_fetch(ctx, h_seg_first, g->seg_first.p, sizeof(uint64_t) * ((size_t)g->nscaf + 1)));
	if(h_seg_scaf)
		ABW_CUDA(ctx, abw_fetch(ctx, h_seg_scaf, g->seg_scaf.p, sizeof(uint32_t) * g->nseg));
	if(h_seg_start)
		ABW_CUDA(ctx, abw_fetch(ctx, h_seg_start, g->seg_start.p, sizeof(uint64_t) * g->nseg));
	if(h_seg_end)
		ABW_CUDA(ctx, abw_fetch(ctx, h_seg_end, g->seg_end.p, sizeof(uint64_t) * g->nseg));
	if(h_seg_nonN)
		ABW_CUDA(ctx, abw_fetch(ctx, h_seg_nonN, g->seg_nonN.p, sizeof(uint64_t) * g->nseg));
	ABW_CUDA(ctx, abw_sync(ctx));
	return ABW_OK;
}

int abw_segments_get_async(abw_ctx* ctx, const abw_segments* g, uint32_t* h_seg_scaf, uint64_t* h_seg_start, uint64_t* h_seg_end, uint64_t* h_seg_nonN)
{
	if(!ctx || !g)
		return abw_fail(ctx, ABW_ERR_ARG, "abw_segments_get_async: null argument");
	if(h_seg_scaf)
		ABW_CHECK(abw_d2h_async(ctx, h_seg_scaf, g->seg_scaf.p, sizeof(uint32_t) * g->nseg));
	if(h_seg_start)
		ABW_CHECK(abw_d2h_async(ctx, h_seg_start, g->seg_start.p, sizeof(uint64_t) * g->nseg));
	if(h_seg_end)
		ABW_CHECK(abw_d2h_async(ctx, h_seg_end, g->seg_end.p, sizeof(uint64_t) * g->nseg));
	if(h_seg_nonN)
		ABW_CHECK(abw_d2h_async(ctx, h_seg_nonN, g->seg_nonN.p, sizeof(uint64_t) * g->nseg));
	return ABW_OK;
}

int abw_kmer_features(abw_ctx* ctx, const abw_seqset* s, const abw_segments* g, int kind, int skip_A, double* d_rows, uint64_t ld, uint32_t col0)
{
	if(!ctx || !s || !g || !d_rows)
		return abw_fail(ctx, ABW_ERR_ARG, "abw_kmer_features: null argument");
	if(kind != ABW_FEAT_TRUNC3 && kind != ABW_FEAT_RAW)
		return abw_fail(ctx, ABW_ERR_ARG, "abw_kmer_features: unknown kind");
	if(ld < (uint64_t)col0 + ABW_NKMER_DIMS - (skip_A? 1 : 0))
		return abw_fail(ctx, ABW_ERR_ARG, "abw_kmer_features: row stride too small");
	ABW_ENTER(ctx);
	ABW_CHECK(upload_tables(ctx));
	if(g->nseg == 0)
		return ABW_OK;
	unsigned int blocks = (unsigned int)std::min<uint64_t>(abw_div_up(g->nseg, KM_WARPS), (uint64_t)ctx->sm_count * 5 * 4);
	if(kind == ABW_FEAT_TRUNC3)
		ABW_LAUNCH(ctx, k_kmer<ABW_FEAT_TRUNC3>, blocks, KM_WARPS * 32, 0, s->packed.p, s->valid.p, g->seg_gbase.p, g->seg_start.p, g->seg_end.p, g->nseg, skip_A, d_rows, ld, col0);
	else
		ABW_LAUNCH(ctx, k_kmer<ABW_FEAT_RAW>, blocks, KM_WARPS * 32, 0, s->packed.p, s->valid.p, g->seg_gbase.p, g->seg_start.p, g->seg_end.p, g->nseg, skip_A, d_rows, ld, col0);
	return ABW_OK;
}

}  // extern "C"
