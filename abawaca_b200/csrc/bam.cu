// BAM files -> read records on the device: the counterpart of abw_parse_sam for the binary format aligner pipelines leave behind.
//
// A BAM file is a series of BGZF blocks (gzip members of at most 64 KiB, each a raw DEFLATE stream whose uncompressed size ISIZE and CRC-32
// are in its trailer).  Per abw_bam_feed:
//  1. the host walks the 18-byte headers and 8-byte trailers of the complete blocks in hand; a running sum of ISIZE gives every block its
//     place in the decoded stream, so the blocks are independent work items;
//  2. k_bgzf_inflate decodes them, one warp per block (inflate.cuh; lane 0 decodes, the warp checks the CRC-32), in batches whose summed ISIZE
//     is at most BATCH_BYTES whatever the compression ratio;
//  3. records may cross block boundaries (htsjdk does not start a block at a record), so their starts are found from the stream: every byte
//     position whose fixed fields describe a well-formed complete record is a candidate, next(p) = p + 4 + block_size, and the records are the
//     chain of candidates from the known first record start, marked by pointer doubling (log2(candidates) rounds);
//  4. one thread per marked record writes its abw_read (the MD walk and the name probe of k_sam_parse, reads.cuh).
// The decoded bytes after the last complete record (and an unfinished header) are carried into the next batch; so is at most one compressed
// block that the feed cut.
#include "common.cuh"
#include "reads.cuh"
#include "inflate.cuh"
#include <algorithm>
#include <cstring>
#include <string>
#include <vector>

namespace {

constexpr uint64_t BATCH_BYTES = (uint64_t)64 << 20;    // decoded bytes per batch (sum of ISIZE)
constexpr int INF_WARPS = 4;                            // decoders per CTA: 4 x 3.6 KB of tables + the CRC table

struct BlockDesc {
	uint64_t cdata;      // offset of the DEFLATE data in the batch's compressed buffer
	uint64_t out;        // offset of the decoded bytes in the batch's stream
	uint32_t clen, isize, crc, pad;
};

constexpr int BAM_ERR_INFLATE = 1, BAM_ERR_CRC = 2, BAM_ERR_AUX = 4, BAM_ERR_MDZ = 8;

__global__ void __launch_bounds__(INF_WARPS * 32, 8) k_bgzf_inflate(const uint8_t* __restrict__ comp, const BlockDesc* __restrict__ blk, uint32_t nblk,
                                                                 uint8_t* __restrict__ out, int* __restrict__ err, uint32_t* __restrict__ err_blk)
{
	abw_grid_wait();
	__shared__ abw_inflate::Tables tables[INF_WARPS];
	__shared__ uint32_t crc_table[256];
	for(int i = threadIdx.x; i < 256; i += blockDim.x)
		crc_table[i] = abw_inflate::crc32_table_entry((uint32_t)i);
	__syncthreads();
	const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
	for(uint32_t b = blockIdx.x * INF_WARPS + warp; b < nblk; b += gridDim.x * INF_WARPS) {
		const BlockDesc d = blk[b];
		uint8_t* o = out + d.out;
		int rc = 0;
		uint32_t olen = 0;
		if(lane == 0)
			rc = abw_inflate::inflate_raw(comp + d.cdata, d.clen, o, d.isize, &olen, tables[warp]);
		rc = __shfl_sync(0xffffffffu, rc, 0);
		olen = __shfl_sync(0xffffffffu, olen, 0);
		__syncwarp();
		int bad = (rc != 0 || olen != d.isize)? BAM_ERR_INFLATE : 0;
		if(!bad) {
			// CRC-32: every lane one slice, combined pairwise
			const uint32_t seg = (d.isize + 31) / 32;
			const uint32_t a = min(d.isize, lane * seg), e = min(d.isize, a + seg);
			uint32_t crc = abw_inflate::crc32(o + a, e - a, crc_table);
			uint32_t len = e - a;
			for(int off = 1; off < 32; off <<= 1) {
				const uint32_t c2 = __shfl_down_sync(0xffffffffu, crc, off), l2 = __shfl_down_sync(0xffffffffu, len, off);
				if((lane & (2 * off - 1)) == 0) {
					crc = abw_inflate::crc32_combine(crc, c2, l2);
					len += l2;
				}
			}
			if(lane == 0 && crc != d.crc)
				bad = BAM_ERR_CRC;
		}
		if(lane == 0 && bad) {
			atomicOr(err, bad);
			atomicMin(err_blk, b);
		}
	}
}

__host__ __device__ __forceinline__ uint32_t ld_u32le(const uint8_t* p) { return (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24); }
__host__ __device__ __forceinline__ uint32_t ld_u16le(const uint8_t* p) { return (uint32_t)p[0] | ((uint32_t)p[1] << 8); }

// The 36 fixed bytes of a record (block_size, then r = the 32 bytes after it) are those of a well-formed record: block_size is an int32 of at least
// 32, refID and next refID are in [-1, n_ref), the name has at least its NUL, and name, CIGAR, SEQ and QUAL fit into block_size.
__host__ __device__ __forceinline__ bool fixed_fields_ok(uint32_t bs, const uint8_t* r, int32_t n_ref)
{
	const int32_t ref = (int32_t)ld_u32le(r), mref = (int32_t)ld_u32le(r + 20), lseq = (int32_t)ld_u32le(r + 16);
	const uint32_t lrn = r[8], ncig = ld_u16le(r + 12);
	return bs >= 32 && bs <= 0x7FFFFFFFu && ref >= -1 && ref < n_ref && mref >= -1 && mref < n_ref && lrn >= 1 && lseq >= 0 &&
	       32ull + lrn + 4ull * ncig + ((uint64_t)lseq + 1) / 2 + (uint64_t)lseq <= bs;
}

// 1 where a complete record whose fixed fields agree with its block_size starts at position p (relative to `start`)
__global__ void k_bam_candidates(const uint8_t* __restrict__ s, uint64_t start, uint64_t len, int32_t n_ref, uint32_t* __restrict__ cand)
{
	abw_grid_wait();
	const uint64_t n = len - start;
	for(uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
		const uint64_t p = start + i;
		uint32_t ok = 0;
		if(p + 36 <= len) {
			const uint32_t bs = ld_u32le(s + p);
			const uint8_t* r = s + p + 4;
			ok = p + 4 + bs <= len && fixed_fields_ok(bs, r, n_ref) && r[32 + r[8] - 1] == 0;
		}
		cand[i] = ok;
	}
}

constexpr uint32_t NXT_END = 0xFFFFFFFFu;      // the record ends exactly at the end of the stream
constexpr uint32_t NXT_LAST = 0xFFFFFFFEu;     // the next position holds no complete candidate: a tail, or the stream is malformed

// candidate positions in order, and each one's successor as a candidate index
__global__ void k_bam_links(const uint8_t* __restrict__ s, uint64_t start, uint64_t len, const uint32_t* __restrict__ cand, const uint64_t* __restrict__ idx,
                            uint64_t* __restrict__ pos, uint32_t* __restrict__ nxt)
{
	abw_grid_wait();
	const uint64_t n = len - start;
	for(uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
		if(!cand[i])
			continue;
		const uint64_t p = start + i, k = idx[i];
		const uint64_t q = p + 4 + ld_u32le(s + p);
		pos[k] = p;
		nxt[k] = (q == len)? NXT_END : cand[q - start]? (uint32_t)idx[q - start] : NXT_LAST;
	}
}

// one pointer-doubling round: successors of marked nodes are marked, jumps double.  Before round k the nodes 0 .. 2^k - 1 steps from the start are
// marked, after it those up to 2^(k+1) - 1 (a node marked early by a concurrent thread is on the chain too, so that race only adds chain nodes).
__global__ void k_bam_chain_round(const uint32_t* __restrict__ jin, uint32_t* __restrict__ jout, uint32_t* mark, uint32_t m)
{
	abw_grid_wait();
	for(uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < m; i += gridDim.x * blockDim.x) {
		const uint32_t j = jin[i];
		if(j < m && mark[i])
			mark[j] = 1;
		jout[i] = (j < m)? jin[j] : j;
	}
}

struct RecArgs {
	const uint8_t* s;
	const uint64_t* pos;
	const uint32_t* mark;
	const uint64_t* slot;
	const uint32_t* nxt;
	uint32_t m;
	const uint32_t* ref_scaf;     // [n_ref + 1]: scaffold of refID r, entry n_ref for refID -1 (RNAME "*")
	int32_t n_ref;
	abw_read* out;
	int* err;
	unsigned long long* after_last;   // where the record after the last marked one starts
};

// one thread per marked record: the abw_read abw_parse_sam makes of the line `samtools view` prints for it
__global__ void __launch_bounds__(128) k_bam_records(RecArgs a)
{
	abw_grid_wait();
	for(uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < a.m; i += gridDim.x * blockDim.x) {
		if(!a.mark[i])
			continue;
		const uint64_t p = a.pos[i];
		const uint8_t* r = a.s + p + 4;
		const uint8_t* end = r + ld_u32le(a.s + p);
		if(a.nxt[i] >= NXT_LAST)
			*a.after_last = (unsigned long long)(end - a.s);
		const int32_t ref = (int32_t)ld_u32le(r), pos = (int32_t)ld_u32le(r + 4);
		const uint32_t lrn = r[8], ncig = ld_u16le(r + 12), flag = ld_u16le(r + 14), lseq = ld_u32le(r + 16);
		const uint8_t* cigar = r + 32 + lrn;
		const uint8_t* q = cigar + 4ull * ncig + ((uint64_t)lseq + 1) / 2 + lseq;     // the aux fields
		// aux fields: the first whose printed text holds "MD:Z:" (only a Z field can), and the first tag named CG
		const char* md = nullptr;
		const char* md_end = nullptr;
		const uint8_t* cg = nullptr;
		uint32_t cg_n = 0;
		bool seen_cg = false, bad = false;
		while(q < end) {
			if(end - q < 3) {
				bad = true;
				break;
			}
			const uint8_t t0 = q[0], t1 = q[1], type = q[2];
			const uint8_t* v = q + 3;
			const uint8_t* next;
			if(type == 'A' || type == 'c' || type == 'C')
				next = v + 1;
			else if(type == 's' || type == 'S')
				next = v + 2;
			else if(type == 'i' || type == 'I' || type == 'f')
				next = v + 4;
			else if(type == 'Z' || type == 'H') {
				const uint8_t* z = v;
				while(z < end && *z)
					z++;
				if(z == end) {
					bad = true;
					break;
				}
				next = z + 1;
				if(type == 'Z' && !md) {
					const char* b = (const char*)v;
					const char* e = (const char*)z;
					if(t0 == 'M' && t1 == 'D')
						md = b;
					else
						for(const char* c = b; c + 5 <= e; c++)
							if(c[0] == 'M' && c[1] == 'D' && c[2] == ':' && c[3] == 'Z' && c[4] == ':') {
								md = c + 5;
								break;
							}
					if(md) {
						md_end = md;
						while(md_end < e && *md_end != ' ')
							md_end++;
					}
				}
			}
			else if(type == 'B') {
				if(end - v < 5) {
					bad = true;
					break;
				}
				const uint8_t sub = v[0];
				const uint32_t cnt = ld_u32le(v + 1);
				const uint32_t es = (sub == 'c' || sub == 'C')? 1 : (sub == 's' || sub == 'S')? 2 : (sub == 'i' || sub == 'I' || sub == 'f')? 4 : 0;
				if(es == 0 || (uint64_t)cnt * es > (uint64_t)(end - (v + 5))) {
					bad = true;
					break;
				}
				if(t0 == 'C' && t1 == 'G' && !seen_cg && (sub == 'I' || sub == 'i')) {
					cg = v + 5;
					cg_n = cnt;
				}
				next = v + 5 + (uint64_t)cnt * es;
			}
			else {
				bad = true;
				break;
			}
			if(next > end) {
				bad = true;
				break;
			}
			if(t0 == 'C' && t1 == 'G')
				seen_cg = true;
			q = next;
		}
		int e = bad? BAM_ERR_AUX : 0;
		uint32_t nsnps = 0;
		if(md && !bad) {
			if(!abw_md_snps(md, md_end, &nsnps))
				e |= BAM_ERR_MDZ;
			// the CIGAR samtools prints: the CG tag's when the record uses the long-CIGAR convention (htslib bam_tag2cigar)
			const bool long_cigar = cg && ncig >= 1 && ref >= 0 && pos >= 0 && (ld_u32le(cigar) & 0xFu) == 4u && (ld_u32le(cigar) >> 4) == lseq;
			const uint8_t* ops = long_cigar? cg : cigar;
			const uint32_t nops = long_cigar? cg_n : ncig;
			uint32_t ins = 0;
			for(uint32_t k = 0; k < nops; k++)
				ins += (ops[4 * k] & 0xFu) == 1u;
			nsnps += ins;
		}
		if(nsnps > 0xFFFFu)
			nsnps = 0xFFFFu;
		abw_read rec;
		rec.scaf = a.ref_scaf[ref < 0? a.n_ref : ref];
		rec.pos0 = (uint32_t)pos;
		rec.len = lseq? lseq : 1u;                 // SAM prints SEQ as "*" when there is none
		rec.flag_nsnps = flag | (nsnps << 16);
		a.out[a.slot[i]] = rec;
		if(e)
			atomicOr(a.err, e);
	}
}

// scaffold index of every reference name of the header (and of "*" for refID -1)
__global__ void k_bam_ref_names(const char* __restrict__ blob, const uint64_t* __restrict__ off, uint32_t n, const unsigned long long* __restrict__ slot_hash,
                                const uint32_t* __restrict__ slot_index, uint32_t nslots, const char* __restrict__ name_blob, const uint64_t* __restrict__ name_off,
                                uint32_t* __restrict__ ref_scaf)
{
	abw_grid_wait();
	const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
	if(i < n)
		ref_scaf[i] = abw_name_probe(blob + off[i], off[i + 1] - off[i], slot_hash, slot_index, nslots, name_blob, name_off);
}

inline uint32_t rd32(const uint8_t* p) { uint32_t v; memcpy(&v, p, 4); return v; }
inline uint32_t rd16(const uint8_t* p) { return (uint32_t)p[0] | ((uint32_t)p[1] << 8); }

// BGZF member header (RFC 1952 with the BC extra subfield): total block size, or 0 when the bytes are not such a header
inline uint32_t bgzf_block_size(const uint8_t* h)
{
	if(h[0] != 31 || h[1] != 139 || h[2] != 8 || h[3] != 4 || rd16(h + 10) != 6 || h[12] != 'B' || h[13] != 'C' || rd16(h + 14) != 2)
		return 0;
	return rd16(h + 16) + 1;
}

template <typename T>
void swap_buf(DevBuf<T>& a, DevBuf<T>& b)
{
	std::swap(a.p, b.p);
	std::swap(a.n, b.n);
	std::swap(a.owner, b.owner);
}

}  // namespace

struct abw_bam {
	const abw_names* names = nullptr;
	std::vector<uint8_t> pending;        // a compressed block the last feed cut
	uint64_t blocks_seen = 0;            // complete blocks so far (for messages)
	DevBuf<uint8_t> stream;              // the last batch's decoded bytes; stream[carry_at .. carry_at + carry) go into the next batch: an unfinished
	uint64_t carry = 0, carry_at = 0;    // header or record
	uint64_t carry_need = 0;             // bytes the carried record or header needs at least before it can be complete (0: not known)
	bool have_header = false;
	int32_t n_ref = 0;
	DevBuf<uint32_t> ref_scaf;
	DevBuf<abw_read> reads;
	uint64_t nreads = 0;
	bool failed = false;
};

namespace {

// The header: magic, l_text, text, n_ref, then n_ref times (l_name, name, l_ref).  Returns its size, 0 while more bytes are needed (*need: a size
// the header cannot be complete below), -1 when malformed.  names gets the reference names as the text prints them (up to the first NUL).
int64_t parse_header(const uint8_t* h, uint64_t n, uint64_t* need, std::string* blob, std::vector<uint64_t>* off)
{
	auto more = [&](uint64_t k) { *need = k; return (int64_t)0; };
	if(n < 12)
		return more(12);
	if(memcmp(h, "BAM\1", 4) != 0)
		return -1;
	const int32_t l_text = (int32_t)rd32(h + 4);
	if(l_text < 0)
		return -1;
	uint64_t p = 8 + (uint64_t)l_text;
	if(n < p + 4)
		return more(p + 4);
	const int32_t n_ref = (int32_t)rd32(h + p);
	if(n_ref < 0)
		return -1;
	p += 4;
	blob->clear();
	off->assign(1, 0);
	for(int32_t i = 0; i < n_ref; i++) {
		if(n < p + 4)
			return more(p + 4);
		const int32_t l_name = (int32_t)rd32(h + p);
		if(l_name < 1)
			return -1;
		if(n < p + 4 + (uint64_t)l_name + 4)
			return more(p + 4 + (uint64_t)l_name + 4);
		const char* nm = (const char*)h + p + 4;
		blob->append(nm, strnlen(nm, (size_t)l_name));
		off->push_back(blob->size());
		p += 4 + (uint64_t)l_name + 4;
	}
	return (int64_t)p;
}

// decode the blocks [0, nblk) whose DEFLATE data is in d_comp and append their records
int run_batch(abw_ctx* ctx, abw_bam* b, const uint8_t* d_comp, const std::vector<BlockDesc>& blk, uint64_t first_block)
{
	const uint32_t nblk = (uint32_t)blk.size();
	const uint64_t decoded = blk.empty()? 0 : blk.back().out + blk.back().isize;
	const uint64_t len = b->carry + decoded;
	DevBuf<uint8_t> s;
	DevBuf<BlockDesc> d_blk;
	DevBuf<int> d_err;
	DevBuf<uint32_t> d_err_blk;
	ABW_CUDA(ctx, s.alloc(len + 64));
	ABW_CUDA(ctx, d_blk.alloc(std::max<uint32_t>(nblk, 1)));
	ABW_CUDA(ctx, d_err.alloc(1));
	ABW_CUDA(ctx, d_err_blk.alloc(1));
	if(b->carry)
		ABW_CUDA(ctx, cudaMemcpyAsync(s.p, b->stream.p + b->carry_at, b->carry, cudaMemcpyDeviceToDevice, ctx->stream));
	ABW_CUDA(ctx, cudaMemsetAsync(d_err.p, 0, sizeof(int), ctx->stream));
	ABW_CUDA(ctx, cudaMemsetAsync(d_err_blk.p, 0xFF, sizeof(uint32_t), ctx->stream));
	if(nblk) {
		ABW_CUDA(ctx, cudaMemcpyAsync(d_blk.p, blk.data(), sizeof(BlockDesc) * nblk, cudaMemcpyHostToDevice, ctx->stream));
		const unsigned int grid = (unsigned int)std::min<uint64_t>(abw_div_up(nblk, INF_WARPS), (uint64_t)ctx->sm_count * 16);
		ABW_LAUNCH(ctx, k_bgzf_inflate, grid, INF_WARPS * 32, 0, d_comp, d_blk.p, nblk, s.p + b->carry, d_err.p, d_err_blk.p);
	}
	int h_err = 0;
	uint32_t h_err_blk = 0;
	ABW_CUDA(ctx, abw_fetch(ctx, &h_err, d_err.p, sizeof(int)));
	ABW_CUDA(ctx, abw_fetch(ctx, &h_err_blk, d_err_blk.p, sizeof(uint32_t)));
	ABW_CUDA(ctx, abw_sync(ctx));
	if(h_err & (BAM_ERR_INFLATE | BAM_ERR_CRC))
		return abw_fail(ctx, ABW_ERR_ARG, std::string("abw_bam_feed: BGZF block ") + std::to_string(first_block + h_err_blk) + " of the file: " +
		                            ((h_err & BAM_ERR_INFLATE)? "invalid DEFLATE data, or not ISIZE bytes of it" : "CRC-32 mismatch"));
	// the carried bytes (start at 0) are an unfinished header or record that cannot be complete yet: nothing to look at
	const bool waiting = len < b->carry_need;
	uint64_t start = 0;
	if(!b->have_header) {
		// the header is parsed on the host from the first bytes of the stream, fetched as far as it needs; the prefix fetched at least doubles
		// every round, so a header is copied and parsed O(log size) times and never more than twice its size is copied
		std::vector<uint8_t> h;
		std::string blob;
		std::vector<uint64_t> off;
		uint64_t need = 0;
		int64_t H = 0;
		for(uint64_t k = waiting? len : std::min<uint64_t>(len, 1 << 16); !waiting;) {
			h.resize(k);
			if(k) {
				ABW_CUDA(ctx, cudaMemcpyAsync(h.data(), s.p, k, cudaMemcpyDeviceToHost, ctx->stream));
				ABW_CUDA(ctx, abw_sync(ctx));
			}
			H = parse_header(h.data(), k, &need, &blob, &off);
			if(H < 0)
				return abw_fail(ctx, ABW_ERR_ARG, "abw_bam_feed: not a BAM file (bad magic) or a malformed BAM header");
			if(H > 0 || k == len)
				break;
			k = std::min(len, std::max(need, 2 * k));
		}
		if(H == 0) {
			swap_buf(b->stream, s);                 // the header is not complete yet: carry all of it
			b->carry = len;
			b->carry_at = 0;
			b->carry_need = std::max(b->carry_need, need);
			return ABW_OK;
		}
		b->have_header = true;
		b->n_ref = (int32_t)(off.size() - 1);
		blob += "*";                                // refID -1 prints RNAME "*", looked up like any name
		off.push_back(blob.size());
		const uint32_t nn = (uint32_t)off.size() - 1;
		DevBuf<char> d_blob;
		DevBuf<uint64_t> d_off;
		ABW_CUDA(ctx, d_blob.alloc(blob.size()));
		ABW_CUDA(ctx, d_off.alloc(off.size()));
		ABW_CUDA(ctx, b->ref_scaf.alloc(nn));
		ABW_CUDA(ctx, cudaMemcpyAsync(d_blob.p, blob.data(), blob.size(), cudaMemcpyHostToDevice, ctx->stream));
		ABW_CUDA(ctx, cudaMemcpyAsync(d_off.p, off.data(), sizeof(uint64_t) * off.size(), cudaMemcpyHostToDevice, ctx->stream));
		const abw_names* nm = b->names;
		ABW_LAUNCH(ctx, k_bam_ref_names, abw_div_up(nn, 128), 128, 0, d_blob.p, d_off.p, nn, nm->slot_hash.p, nm->slot_index.p, nm->nslots, nm->blob.p, nm->off.p,
		           b->ref_scaf.p);
		ABW_CUDA(ctx, abw_sync(ctx));              // blob and off are locals
		start = (uint64_t)H;
	}
	const uint64_t n = len - start;
	const int grid = (int)std::min<uint64_t>(std::max<uint64_t>(abw_div_up(n, 256), 1), (uint64_t)ctx->sm_count * 32);
	uint64_t m = 0, after_last = start;
	if(n >= 36 && !(waiting && start == 0)) {
		DevBuf<uint32_t> cand;
		DevBuf<uint64_t> idx, total;
		ABW_CUDA(ctx, cand.alloc(n));
		ABW_CUDA(ctx, idx.alloc(n));
		ABW_CUDA(ctx, total.alloc(2));
		ABW_LAUNCH(ctx, k_bam_candidates, grid, 256, 0, s.p, start, len, b->n_ref, cand.p);
		ABW_CHECK(abw_exclusive_scan_u32_to_u64(ctx, cand.p, idx.p, n, total.p));
		uint32_t c0 = 0;
		ABW_CUDA(ctx, abw_fetch(ctx, &m, total.p, sizeof(uint64_t)));
		ABW_CUDA(ctx, abw_fetch(ctx, &c0, cand.p, sizeof(uint32_t)));
		ABW_CUDA(ctx, abw_sync(ctx));
		if(m >= NXT_LAST)
			return abw_fail(ctx, ABW_ERR_UNSUPPORTED, "abw_bam_feed: too many record candidates in one batch");
		if(c0) {
			// the chain from the first record start (candidate 0)
			DevBuf<uint64_t> pos, slot;
			DevBuf<uint32_t> nxt, ja, jb, mark;
			ABW_CUDA(ctx, pos.alloc(m));
			ABW_CUDA(ctx, nxt.alloc(m));
			ABW_CUDA(ctx, ja.alloc(m));
			ABW_CUDA(ctx, jb.alloc(m));
			ABW_CUDA(ctx, mark.alloc(m));
			ABW_CUDA(ctx, slot.alloc(m));
			ABW_LAUNCH(ctx, k_bam_links, grid, 256, 0, s.p, start, len, cand.p, idx.p, pos.p, nxt.p);
			ABW_CUDA(ctx, cudaMemsetAsync(mark.p, 0, sizeof(uint32_t) * m, ctx->stream));
			const uint32_t one = 1;
			ABW_CUDA(ctx, cudaMemcpyAsync(mark.p, &one, sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
			const unsigned int mg = std::min<uint64_t>(abw_div_up(m, 256), (uint64_t)ctx->sm_count * 32);
			const uint32_t* jin = nxt.p;
			uint32_t* jout = ja.p;
			for(uint64_t reach = 1; reach < m; reach <<= 1) {
				ABW_LAUNCH(ctx, k_bam_chain_round, mg, 256, 0, jin, jout, mark.p, (uint32_t)m);
				jin = jout;
				jout = (jout == ja.p)? jb.p : ja.p;
			}
			uint64_t nrec = 0;
			ABW_CHECK(abw_exclusive_scan_u32_to_u64(ctx, mark.p, slot.p, m, total.p + 1));
			ABW_CUDA(ctx, abw_fetch(ctx, &nrec, total.p + 1, sizeof(uint64_t)));
			ABW_CUDA(ctx, abw_sync(ctx));           // `one` is a local
			if(b->nreads + nrec > b->reads.n) {
				DevBuf<abw_read> grown;
				ABW_CUDA(ctx, grown.alloc(std::max<uint64_t>(2 * b->reads.n, b->nreads + nrec)));
				if(b->nreads)
					ABW_CUDA(ctx, cudaMemcpyAsync(grown.p, b->reads.p, sizeof(abw_read) * b->nreads, cudaMemcpyDeviceToDevice, ctx->stream));
				swap_buf(b->reads, grown);
			}
			DevBuf<unsigned long long> d_after;
			ABW_CUDA(ctx, d_after.alloc(1));
			ABW_CUDA(ctx, cudaMemsetAsync(d_err.p, 0, sizeof(int), ctx->stream));
			RecArgs ra{s.p, pos.p, mark.p, slot.p, nxt.p, (uint32_t)m, b->ref_scaf.p, b->n_ref, b->reads.p + b->nreads, d_err.p, d_after.p};
			ABW_LAUNCH(ctx, k_bam_records, (unsigned int)std::min<uint64_t>(abw_div_up(m, 128), (uint64_t)ctx->sm_count * 64), 128, 0, ra);
			ABW_CUDA(ctx, abw_fetch(ctx, &h_err, d_err.p, sizeof(int)));
			ABW_CUDA(ctx, abw_fetch(ctx, &after_last, d_after.p, sizeof(uint64_t)));
			ABW_CUDA(ctx, abw_sync(ctx));
			if(h_err & BAM_ERR_AUX)
				return abw_fail(ctx, ABW_ERR_ARG, "abw_bam_feed: a BAM record's aux fields do not parse to the end of the record");
			if(h_err & BAM_ERR_MDZ)
				return abw_fail(ctx, ABW_ERR_ARG, "abw_parse_sam: Illegal SNPs description in an MD:Z field (Illegal_mapping, ReadMapping.cpp:100-113)");
			b->nreads += nrec;
		}
	}
	// after_last: where the record after the last one found starts; from there on the bytes must be an unfinished record, and its fixed fields,
	// as far as they are there, those of a well-formed record
	b->carry_need = 0;
	if(after_last < len) {
		uint8_t f[36];
		const uint64_t k = std::min<uint64_t>(36, len - after_last);
		ABW_CUDA(ctx, cudaMemcpyAsync(f, s.p + after_last, k, cudaMemcpyDeviceToHost, ctx->stream));
		ABW_CUDA(ctx, abw_sync(ctx));
		if(k >= 4) {
			const uint32_t bs = rd32(f);
			if(bs < 32 || bs > 0x7FFFFFFFu || after_last + 4 + bs <= len || (k == 36 && !fixed_fields_ok(bs, f + 4, b->n_ref)))
				return abw_fail(ctx, ABW_ERR_ARG, "abw_bam_feed: a BAM record's block_size disagrees with its fixed fields");
			b->carry_need = 4 + (uint64_t)bs;
		}
	}
	b->carry = len - after_last;
	b->carry_at = after_last;
	swap_buf(b->stream, s);
	return ABW_OK;
}

}  // namespace

extern "C" {

int abw_bam_create(abw_ctx* ctx, const abw_names* names, abw_bam** out)
{
	if(!ctx || !names || !out)
		return abw_fail(ctx, ABW_ERR_ARG, "abw_bam_create: null argument");
	*out = new abw_bam();
	(*out)->names = names;
	return ABW_OK;
}

void abw_bam_destroy(abw_bam* b) { delete b; }

}  // extern "C"

namespace {

int bam_feed(abw_ctx* ctx, abw_bam* b, const uint8_t* data, uint64_t nbytes)
{
	uint64_t at = 0;
	auto bad_header = [&]() { return abw_fail(ctx, ABW_ERR_ARG, "abw_bam_feed: BGZF block " + std::to_string(b->blocks_seen) + " of the file: not a BGZF block header"); };
	// complete the block the previous feed cut
	bool have_pending_block = false;
	if(!b->pending.empty()) {
		if(b->pending.size() < 18) {
			const uint64_t k = std::min<uint64_t>(18 - b->pending.size(), nbytes);
			b->pending.insert(b->pending.end(), data, data + k);
			at = k;
		}
		if(b->pending.size() >= 18) {
			const uint32_t bsize = bgzf_block_size(b->pending.data());
			if(bsize < 26)
				return bad_header();
			const uint64_t k = std::min<uint64_t>(bsize - b->pending.size(), nbytes - at);
			b->pending.insert(b->pending.end(), data + at, data + at + k);
			at += k;
			have_pending_block = b->pending.size() == bsize;
		}
		if(!have_pending_block)
			return ABW_OK;
	}
	// the complete blocks of this feed
	struct Span { const uint8_t* p; uint32_t size; };
	std::vector<Span> blocks;
	if(have_pending_block)
		blocks.push_back({b->pending.data(), (uint32_t)b->pending.size()});
	while(nbytes - at >= 18) {
		const uint32_t bsize = bgzf_block_size(data + at);
		if(bsize < 26) {
			b->blocks_seen += blocks.size();
			return bad_header();
		}
		if(bsize > nbytes - at)
			break;
		blocks.push_back({data + at, bsize});
		at += bsize;
	}
	// batches of blocks of at most BATCH_BYTES decoded bytes
	DevBuf<uint8_t> comp;
	size_t i = 0;
	while(i < blocks.size()) {
		std::vector<BlockDesc> desc;
		uint64_t out = 0, cbytes = 0;
		size_t j = i;
		for(; j < blocks.size(); j++) {
			const Span& sp = blocks[j];
			const uint32_t isize = rd32(sp.p + sp.size - 4);
			if(isize > 65536)
				return abw_fail(ctx, ABW_ERR_ARG, "abw_bam_feed: BGZF block " + std::to_string(b->blocks_seen + j) + " of the file: ISIZE above 65536");
			if(j > i && out + isize > BATCH_BYTES)
				break;
			desc.push_back({cbytes, out, sp.size - 26, isize, rd32(sp.p + sp.size - 8), 0});
			out += isize;
			cbytes += sp.size;
		}
		ABW_CUDA(ctx, comp.alloc(cbytes + 16));
		// the blocks of a batch are adjacent in the feed, except a completed pending block, which comes first
		uint64_t c = 0;
		size_t k = i;
		if(k == 0 && have_pending_block) {
			ABW_CUDA(ctx, cudaMemcpyAsync(comp.p, blocks[0].p, blocks[0].size, cudaMemcpyHostToDevice, ctx->stream));
			c = blocks[0].size;
			k = 1;
		}
		if(k < j)
			ABW_CUDA(ctx, cudaMemcpyAsync(comp.p + c, blocks[k].p, cbytes - c, cudaMemcpyHostToDevice, ctx->stream));
		for(BlockDesc& d : desc)
			d.cdata += 18;
		ABW_CHECK(run_batch(ctx, b, comp.p, desc, b->blocks_seen + i));
		i = j;
	}
	b->blocks_seen += blocks.size();
	b->pending.assign(data + at, data + nbytes);
	return ABW_OK;
}

}  // namespace

extern "C" {

int abw_bam_feed(abw_ctx* ctx, abw_bam* b, const void* h_data, uint64_t nbytes)
{
	if(!ctx || !b || (!h_data && nbytes))
		return abw_fail(ctx, ABW_ERR_ARG, "abw_bam_feed: null argument");
	if(b->failed)
		return abw_fail(ctx, ABW_ERR_ARG, "abw_bam_feed: the reader failed on earlier input");
	ABW_ENTER(ctx);
	// any error (malformed input, CUDA, resources) may leave the carried state half updated: the reader takes no further input
	const int rc = bam_feed(ctx, b, (const uint8_t*)h_data, nbytes);
	if(rc != ABW_OK)
		b->failed = true;
	return rc;
}

int abw_bam_finish(abw_ctx* ctx, abw_bam* b, const abw_read** d_reads, uint64_t* nreads)
{
	if(!ctx || !b || !d_reads || !nreads)
		return abw_fail(ctx, ABW_ERR_ARG, "abw_bam_finish: null argument");
	if(b->failed)
		return abw_fail(ctx, ABW_ERR_ARG, "abw_bam_finish: the reader failed on earlier input");
	if(!b->pending.empty())
		return abw_fail(ctx, ABW_ERR_ARG, "abw_bam_finish: the BAM stream ends inside a BGZF block");
	if(!b->have_header)
		return abw_fail(ctx, ABW_ERR_ARG, "abw_bam_finish: the BAM stream ends inside its header");
	if(b->carry)
		return abw_fail(ctx, ABW_ERR_ARG, "abw_bam_finish: the BAM stream ends inside a record");
	*d_reads = b->reads.p;
	*nreads = b->nreads;
	return ABW_OK;
}

}  // extern "C"
