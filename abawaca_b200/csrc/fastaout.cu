// Records -> FASTA text on the device (SURVEY.md section 8f, row 2: the text writers of abawaca).
//
// Replaces SeqIOWrite_fasta as abawaca writes final-clusters/<id>.fasta (abawaca.cpp:141-142): per record "><id> <desc>\n", then the sequence
// upper-cased ("C" locale toupper: only a-z change) in lines of 60 characters, floor(L / 60) + 1 lines, the last one holding L % 60 (possibly none).
//
// The layout is known on the host before any kernel runs (the handles keep every record's id, description and sequence length there), so the host
// numbers the records' first bytes and cuts the caller's window; k_fasta_write then makes the window in one pass.  One thread makes the 16 bytes of
// one 16-byte-aligned ADDRESS range of the output and stores them as one word (single bytes at the window's two ends); consecutive threads make
// consecutive output, so a warp reads about 500 consecutive bytes of text or 125 of .2bit codes.  A thread finds its record by binary search over
// the window's records, its first sequence line (FASTA) or N block (.2bit) by binary search too, and walks on from there.
#include "fastaout.cuh"
#include <algorithm>

namespace {

constexpr uint32_t FA_COLS = 60;

// a window's record with the offset of its first byte in the whole text
struct FaItem {
	FaRecord r;
	uint64_t off;
};

__device__ __forceinline__ uint32_t fa_upper(uint32_t c) { return (c - 'a' < 26u)? c - 32u : c; }

__device__ __forceinline__ uint64_t fa_hdr_len(const FaRecord& r) { return 3ull + r.id_len + r.desc_len; }

template <int KIND>
__global__ void __launch_bounds__(256) k_fasta_write(FaSource src, const FaItem* __restrict__ items, uint32_t nitems, uint64_t byte0, uint64_t n,
                                                     char* __restrict__ out)
{
	abw_grid_wait();
	const char* __restrict__ text = src.text;
	const uintptr_t o0 = reinterpret_cast<uintptr_t>(out), o1 = o0 + n, base = o0 & ~(uintptr_t)15;
	const uint64_t nchunks = (o1 - base + 15) >> 4;
	const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
	for(uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; t < nchunks; t += stride) {
		const uintptr_t a0 = max(base + 16 * t, o0), a1 = min(base + 16 * t + 16, o1);
		uint64_t p = byte0 + (a0 - o0);                                 // position in the whole text
		// the record that holds p: the last item whose offset is <= p
		uint32_t lo = 0, hi = nitems - 1;
		while(lo < hi) {
			const uint32_t mid = (lo + hi + 1) >> 1;
			if(items[mid].off <= p) lo = mid; else hi = mid - 1;
		}
		uint32_t it = lo;
		FaRecord r = items[it].r;
		uint64_t q = p - items[it].off, hdr = fa_hdr_len(r), end = hdr + r.len + r.len / FA_COLS + 1;
		// sequence cursor: line `line` of the record, column `col`; FASTA: text line l holds the record's characters [g0, g1) (global numbering);
		// .2bit: N block `blk`
		bool cur = false;
		uint64_t line = 0, g0 = 1, g1 = 0, ta = 0, blk = 0;
		uint32_t col = 0;
		unsigned long long lo8 = 0, hi8 = 0;                            // the 16 bytes of a full word, in registers
		for(uint32_t j = 0; j < (uint32_t)(a1 - a0); j++, p++, q++) {
			while(q >= end) {                                            // the thread's bytes run into the next record
				it++;
				r = items[it].r;
				q = 0;
				hdr = fa_hdr_len(r);
				end = hdr + r.len + r.len / FA_COLS + 1;
				cur = false;
			}
			uint32_t b;
			if(q < hdr) {
				if(q == 0)
					b = '>';
				else if(q <= r.id_len)
					b = (unsigned char)text[r.id_off + q - 1];
				else if(q == r.id_len + 1ull)
					b = ' ';
				else if(q < hdr - 1)
					b = (unsigned char)text[r.desc_off + (q - r.id_len - 2)];
				else
					b = '\n';
			}
			else {
				if(!cur) {
					const uint64_t s = q - hdr;
					line = s / (FA_COLS + 1);
					col = (uint32_t)(s - line * (FA_COLS + 1));
					cur = true;
					if(KIND == FA_SRC_2BIT) {
						// the first block that ends after the first base this thread may need
						const uint64_t k = line * FA_COLS + min(col, FA_COLS - 1);
						uint64_t bl = r.nb0, bh = r.nb1;
						while(bl < bh) {
							const uint64_t mid = (bl + bh) >> 1;
							const uint2 nb = src.nblocks[mid];
							if((uint64_t)nb.x + nb.y <= k) bl = mid + 1; else bh = mid;
						}
						blk = bl;
					}
					else
						g0 = 1, g1 = 0;                                      // no line yet
				}
				const uint64_t k = line * FA_COLS + col;
				if(col == FA_COLS || k >= r.len)
					b = '\n';
				else if(KIND == FA_SRC_TEXT) {
					const uint64_t g = r.seq0 + k;
					if(g < g0 || g >= g1) {
						// the sequence line that holds character g: the last line with chars_before <= g (it has characters: the next one starts after g)
						uint64_t ll = 0, lh = src.nlines - 1;
						while(ll < lh) {
							const uint64_t mid = (ll + lh + 1) >> 1;
							if(src.chars_before[mid] <= g) ll = mid; else lh = mid - 1;
						}
						g0 = src.chars_before[ll];
						g1 = g0 + src.line_len[ll];
						ta = src.line_a[ll];
					}
					b = fa_upper((unsigned char)text[ta + (g - g0)]);
				}
				else {
					while(blk < r.nb1 && (uint64_t)src.nblocks[blk].x + src.nblocks[blk].y <= k)
						blk++;
					if(blk < r.nb1 && src.nblocks[blk].x <= k)
						b = 'N';
					else
						b = (unsigned char)"TCAG"[((unsigned char)text[r.seq0 + (k >> 2)] >> (6 - 2 * (k & 3))) & 3];
				}
				if(++col > FA_COLS) {
					col = 0;
					line++;
				}
			}
			if(a1 - a0 == 16) {
				if(j < 8)
					lo8 |= (unsigned long long)b << (8 * j);
				else
					hi8 |= (unsigned long long)b << (8 * (j - 8));
			}
			else
				reinterpret_cast<char*>(a0)[j] = (char)b;
		}
		if(a1 - a0 == 16)
			*reinterpret_cast<uint4*>(a0) = make_uint4((uint32_t)lo8, (uint32_t)(lo8 >> 32), (uint32_t)hi8, (uint32_t)(hi8 >> 32));
	}
}

}  // namespace

int abw_fasta_text(abw_ctx* ctx, const FaSource& src, const std::vector<FaRecord>& recs, uint64_t byte0, char* d_text, uint64_t cap, uint64_t* total,
                   uint64_t* nbytes)
{
	// offsets of every record's first byte in the whole text
	const size_t nrecs = recs.size();
	std::vector<uint64_t> off(nrecs + 1, 0);
	for(size_t i = 0; i < nrecs; i++) {
		const FaRecord& r = recs[i];
		off[i + 1] = off[i] + 3 + r.id_len + r.desc_len + r.len + r.len / FA_COLS + 1;
	}
	*total = off[nrecs];
	*nbytes = 0;
	if(byte0 >= off[nrecs] || cap == 0)
		return ABW_OK;
	if(!d_text)
		return abw_fail(ctx, ABW_ERR_ARG, "abw_fasta_format: null text buffer");
	const uint64_t n = std::min(cap, off[nrecs] - byte0);
	// the records the window touches: from the one that holds byte0 to the one that holds its last byte
	const size_t i0 = (size_t)(std::upper_bound(off.begin(), off.end(), byte0) - off.begin()) - 1;
	const size_t i1 = (size_t)(std::upper_bound(off.begin(), off.end(), byte0 + n - 1) - off.begin());
	std::vector<FaItem> items(i1 - i0);
	for(size_t i = i0; i < i1; i++)
		items[i - i0] = FaItem{recs[i], off[i]};
	DevBuf<FaItem> d_items;
	ABW_CUDA(ctx, d_items.alloc(items.size()));
	ABW_CUDA(ctx, abw_upload_small(ctx, d_items.p, items.data(), sizeof(FaItem) * items.size()));
	const uintptr_t o0 = reinterpret_cast<uintptr_t>(d_text);
	const uint64_t nchunks = ((o0 + n + 15) >> 4) - (o0 >> 4);
	const unsigned int blocks = (unsigned int)std::min<uint64_t>(abw_div_up(nchunks, 256), (uint64_t)ctx->sm_count * 32);
	if(src.kind == FA_SRC_TEXT)
		ABW_LAUNCH(ctx, k_fasta_write<FA_SRC_TEXT>, blocks, 256, 0, src, d_items.p, (uint32_t)items.size(), byte0, n, d_text);
	else
		ABW_LAUNCH(ctx, k_fasta_write<FA_SRC_2BIT>, blocks, 256, 0, src, d_items.p, (uint32_t)items.size(), byte0, n, d_text);
	ABW_CUDA(ctx, abw_sync(ctx));      // the item table is a local (and the staging area is free again after the wait)
	*nbytes = n;
	return ABW_OK;
}
