// Text parsers on the device (SURVEY.md section 8f: host text parsing is > 80 % of abawaca-build):
//   SAM    (abw_parse_sam)    -> the abw_read record stream abw_coverage consumes, in file order
//   FASTA  (abw_fasta_scan)   -> records with their ids and trimmed sequence lines, packed by abw_fasta_pack, counted by abw_fasta_base_counts and
//                                written back as abawaca prints them by abw_fasta_format (fastaout.cu)
//   .lrn   (abw_parse_lrn)    -> keys and a row-major matrix of doubles
//
// The three share one line index (line_index): newline positions are counted per 4 KB tile and scanned, which gives every line its index, and a
// second pass writes the line starts.  SAM and .lrn also share one line selection (select_lines): the last byte and the first byte of a line decide
// whether it is a record, and a scan over those flags gives the record its slot.  One thread then parses one line.
//
// For SAM this replaces, for one chunk of text,
//   SAMReader::next_mapping            ReadMappingReader.cpp:80-116  (lines; '@' header lines and empty lines are skipped)
//   ReadMapping::ReadMapping(line)     ReadMapping.cpp:23-72         (tab-separated fields: FLAG, RNAME, POS-1, CIGAR, SEQ, the field holding "MD:Z:")
//   ReadMapping::determine_snps        ReadMapping.cpp:78-185        (only num_snps() reaches the hot path: one per mismatch letter of MD:Z, one per
//                                                                     deleted reference base after '^', one per insertion operation of the CIGAR string)
//   scafs.find(ref_name)               abawaca-build.cpp:549         (reference name -> scaffold index; unknown names give index 0xFFFFFFFF)
#include "common.cuh"
#include "reads.cuh"
#include "fastaout.cuh"
#include <algorithm>
#include <cstring>
#include <cstdlib>
#include <vector>

namespace {

constexpr int LN_THREADS = 256;
constexpr int LN_BYTES_PER_THREAD = 16;
constexpr int LN_TILE = LN_THREADS * LN_BYTES_PER_THREAD;      // 4 KB of text per block

__global__ void __launch_bounds__(LN_THREADS) k_line_count(const char* __restrict__ text, uint64_t nbytes, uint32_t* __restrict__ tile_counts)
{
	abw_grid_wait();
	__shared__ uint32_t sm[LN_THREADS / 32];
	const uint64_t i0 = (uint64_t)blockIdx.x * LN_TILE + (uint64_t)threadIdx.x * LN_BYTES_PER_THREAD;
	uint32_t c = 0;
	if(i0 + LN_BYTES_PER_THREAD <= nbytes && ((reinterpret_cast<uintptr_t>(text + i0) & 15) == 0)) {
		const uint4 w = __ldg(reinterpret_cast<const uint4*>(text + i0));
		c = __popc(__vcmpeq4(w.x, 0x0A0A0A0Au) & 0x01010101u) + __popc(__vcmpeq4(w.y, 0x0A0A0A0Au) & 0x01010101u) +
		    __popc(__vcmpeq4(w.z, 0x0A0A0A0Au) & 0x01010101u) + __popc(__vcmpeq4(w.w, 0x0A0A0A0Au) & 0x01010101u);
	}
	else {
		for(int j = 0; j < LN_BYTES_PER_THREAD; j++)
			if(i0 + j < nbytes && text[i0 + j] == '\n')
				c++;
	}
	c = __reduce_add_sync(0xffffffffu, c);
	if((threadIdx.x & 31) == 0)
		sm[threadIdx.x >> 5] = c;
	__syncthreads();
	if(threadIdx.x == 0) {
		uint32_t t = 0;
		for(int w = 0; w < LN_THREADS / 32; w++)
			t += sm[w];
		tile_counts[blockIdx.x] = t;
	}
}

// line l (l >= 1) starts after the l-th newline; line 0 starts at 0.  A final newline opens an empty last line, which is not a record.
__global__ void __launch_bounds__(LN_THREADS) k_line_starts(const char* __restrict__ text, uint64_t nbytes, const uint64_t* __restrict__ tile_offs, uint64_t* __restrict__ line_start)
{
	abw_grid_wait();
	__shared__ uint32_t sm[LN_THREADS / 32];
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	const uint64_t i0 = (uint64_t)blockIdx.x * LN_TILE + (uint64_t)threadIdx.x * LN_BYTES_PER_THREAD;
	uint32_t mask = 0;
	for(int j = 0; j < LN_BYTES_PER_THREAD; j++)
		if(i0 + j < nbytes && text[i0 + j] == '\n')
			mask |= 1u << j;
	const uint32_t c = __popc(mask);
	uint32_t incl = c;
#pragma unroll
	for(int o = 1; o < 32; o <<= 1) {
		const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
		if(lane >= o)
			incl += t;
	}
	if(lane == 31)
		sm[warp] = incl;
	__syncthreads();
	uint32_t wex = 0;
	for(int w = 0; w < warp; w++)
		wex += sm[w];
	uint64_t rank = tile_offs[blockIdx.x] + wex + incl - c;      // newlines before this thread's bytes
	if(blockIdx.x == 0 && threadIdx.x == 0)
		line_start[0] = 0;
	while(mask) {
		const int j = __ffs(mask) - 1;
		mask &= mask - 1;
		rank++;
		line_start[rank] = i0 + j + 1;
	}
}

// The line index of a text on the device: line l is [start[l], start[l + 1] - 1), the last line ends at nbytes.
struct LineIndex {
	DevBuf<char> staged;                      // the text, when it was given on the host
	const char* text = nullptr;
	uint64_t nbytes = 0, nlines = 0;
	DevBuf<uint64_t> start;
};

// Stages host text (text_on_device == 0) and indexes its lines, with one wait on the context stream for the number of newlines.  nbytes > 0.
int line_index(abw_ctx* ctx, const char* text, uint64_t nbytes, int text_on_device, LineIndex* li)
{
	li->nbytes = nbytes;
	li->text = text;
	if(!text_on_device) {
		ABW_CUDA(ctx, li->staged.alloc(nbytes + 16));
		ABW_CUDA(ctx, cudaMemcpyAsync(li->staged.p, text, nbytes, cudaMemcpyHostToDevice, ctx->stream));
		li->text = li->staged.p;
	}
	const unsigned int ntiles = abw_div_up(nbytes, LN_TILE);
	DevBuf<uint32_t> tile_counts;
	DevBuf<uint64_t> tile_offs, total;
	ABW_CUDA(ctx, tile_counts.alloc(ntiles));
	ABW_CUDA(ctx, tile_offs.alloc(ntiles));
	ABW_CUDA(ctx, total.alloc(1));
	ABW_LAUNCH(ctx, k_line_count, ntiles, LN_THREADS, 0, li->text, nbytes, tile_counts.p);
	ABW_CHECK(abw_exclusive_scan_u32_to_u64(ctx, tile_counts.p, tile_offs.p, ntiles, total.p));
	uint64_t nnl = 0;
	ABW_CUDA(ctx, abw_fetch(ctx, &nnl, total.p, sizeof(uint64_t)));
	ABW_CUDA(ctx, abw_sync(ctx));
	li->nlines = nnl + 1;
	ABW_CUDA(ctx, li->start.alloc(li->nlines));
	ABW_LAUNCH(ctx, k_line_starts, ntiles, LN_THREADS, 0, li->text, nbytes, tile_offs.p, li->start.p);
	return ABW_OK;
}

// [a, b) of line l, without its newline
struct LineExtent { uint64_t a, b; };
__device__ __forceinline__ LineExtent line_extent(const uint64_t* __restrict__ line_start, uint64_t nlines, uint64_t nbytes, uint64_t l)
{
	return {line_start[l], (l + 1 < nlines)? line_start[l + 1] - 1 : nbytes};
}

__device__ __forceinline__ bool dev_isspace(char c) { return c == ' ' || (c >= '\t' && c <= '\r'); }

// 1 for a line that is not empty after trimming its end and does not start with `skip`.  The end is trimmed of all white space (trim_space) or
// only of '\r' and '\n':
//   SAM   ('@', false): chomp (ReadMappingReader.cpp:113) and header lines (:108).  fgets-based reading stops a line at '\n'; a line that is just
//         "\n" or "\r\n" has next_line[0] == '\n' (not 0 and not '@'), so the reference would try to parse it and fail on fs[1]; real SAM files
//         have no such lines and abawaca_b200's host parser skips them, as does this one.  A line of blanks is a record (and too short).
//   .lrn  ('%', true): empty and comment lines (ClusterData.cpp:110-168); a line of blanks is empty.
__global__ void k_line_select(const char* __restrict__ text, uint64_t nbytes, const uint64_t* __restrict__ line_start, uint64_t nlines, char skip, bool trim_space,
                              uint32_t* __restrict__ keep)
{
	abw_grid_wait();
	const uint64_t l = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if(l >= nlines)
		return;
	auto [a, b] = line_extent(line_start, nlines, nbytes, l);
	while(b > a && (trim_space? dev_isspace(text[b - 1]) : (text[b - 1] == '\r' || text[b - 1] == '\n')))
		b--;
	keep[l] = (b > a && text[a] != skip)? 1u : 0u;
}

// Flags the lines k_line_select keeps and numbers them (slot[l] = kept lines before l); *count is the number kept, after one wait.
int select_lines(abw_ctx* ctx, const LineIndex& li, char skip, bool trim_space, DevBuf<uint32_t>& keep, DevBuf<uint64_t>& slot, uint64_t* count)
{
	DevBuf<uint64_t> total;
	ABW_CUDA(ctx, keep.alloc(li.nlines));
	ABW_CUDA(ctx, slot.alloc(li.nlines));
	ABW_CUDA(ctx, total.alloc(1));
	ABW_LAUNCH(ctx, k_line_select, abw_div_up(li.nlines, 256), 256, 0, li.text, li.nbytes, li.start.p, li.nlines, skip, trim_space, keep.p);
	ABW_CHECK(abw_exclusive_scan_u32_to_u64(ctx, keep.p, slot.p, li.nlines, total.p));
	ABW_CUDA(ctx, abw_fetch(ctx, count, total.p, sizeof(uint64_t)));
	ABW_CUDA(ctx, abw_sync(ctx));
	return ABW_OK;
}

// atoi on a field [p, e): optional white space, optional sign, digits (ReadMapping.cpp:39,41 call atoi on the field text)
__device__ __forceinline__ int dev_atoi(const char* __restrict__ p, const char* __restrict__ e)
{
	while(p < e && dev_isspace(*p))
		p++;
	bool neg = false;
	if(p < e && (*p == '+' || *p == '-')) {
		neg = *p == '-';
		p++;
	}
	unsigned int v = 0;
	while(p < e && *p >= '0' && *p <= '9') {
		v = v * 10u + (unsigned int)(*p - '0');
		p++;
	}
	return neg? -(int)v : (int)v;
}

constexpr int SAM_ERR_FEW_FIELDS = 1, SAM_ERR_LOWER_N = 2, SAM_ERR_MDZ = 4;

__global__ void __launch_bounds__(128) k_sam_parse(const char* __restrict__ text, uint64_t nbytes, const uint64_t* __restrict__ line_start, uint64_t nlines,
                                                   const uint32_t* __restrict__ is_record, const uint64_t* __restrict__ rec_slot, const unsigned long long* __restrict__ slot_hash,
                                                   const uint32_t* __restrict__ slot_index, uint32_t nslots, const char* __restrict__ name_blob,
                                                   const uint64_t* __restrict__ name_off, abw_read* __restrict__ out, uint64_t cap, int* __restrict__ err)
{
	abw_grid_wait();
	const uint64_t l = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if(l >= nlines || !is_record[l])
		return;
	const uint64_t slot = rec_slot[l];
	if(slot >= cap)
		return;
	const auto [a, b] = line_extent(line_start, nlines, nbytes, l);
	const char* p = text + a;
	const char* e = text + b;
	while(e > p && (e[-1] == '\r' || e[-1] == '\n'))       // chomp, ReadMappingReader.cpp:113
		e--;
	// walk the tab-separated fields (split('\t', ...), ReadMapping.cpp:36)
	int field = 0;
	const char* fs = p;                                    // start of the current field
	uint32_t flag = 0, scaf = 0xFFFFFFFFu, pos0 = 0, len = 0, nsnps = 0, cigar_ins = 0;
	bool have_md = false;
	int bad = 0;
	for(const char* q = p;; q++) {
		if(q == e || *q == '\t') {
			const char* fe = q;
			if(field == 1)
				flag = (uint32_t)dev_atoi(fs, fe);
			else if(field == 2)
				scaf = abw_name_probe(fs, (uint64_t)(fe - fs), slot_hash, slot_index, nslots, name_blob, name_off);
			else if(field == 3)
				pos0 = (uint32_t)(dev_atoi(fs, fe) - 1);    // stored 0-based, ReadMapping.cpp:41
			else if(field == 5) {
				for(const char* c = fs; c < fe; c++)
					cigar_ins += (*c == 'I');                   // one INSERTION entry per I operation, ReadMapping.cpp:160-173
			}
			else if(field == 9) {
				len = (uint32_t)(fe - fs);                      // SEQ.size(), ReadMapping.h:44
				for(const char* c = fs; c < fe; c++)
					if(*c == 'n')
						bad |= SAM_ERR_LOWER_N;                 // Bio::DNAString throws, String.cpp:47-49
			}
			else if(field >= 11 && !have_md) {
				// the first optional field that contains "MD:Z:" anywhere; the description runs to the first space or the end of the field (:53-66)
				for(const char* c = fs; c + 5 <= fe; c++) {
					if(c[0] == 'M' && c[1] == 'D' && c[2] == ':' && c[3] == 'Z' && c[4] == ':') {
						have_md = true;
						const char* m = c + 5;
						const char* me = m;
						while(me < fe && *me != ' ')
							me++;
						if(!abw_md_snps(m, me, &nsnps))
							bad |= SAM_ERR_MDZ;
						break;
					}
				}
			}
			field++;
			fs = q + 1;
			if(q == e)
				break;
		}
	}
	if(field < 11)
		bad |= SAM_ERR_FEW_FIELDS;                          // fs[10] is read unconditionally, ReadMapping.cpp:51
	if(have_md)
		nsnps += cigar_ins;                                 // without an MD:Z field determine_snps returns at once (:80-81)
	else
		nsnps = 0;
	if(nsnps > 0xFFFFu)
		nsnps = 0xFFFFu;
	abw_read r;
	r.scaf = scaf;
	r.pos0 = pos0;
	r.len = len;
	r.flag_nsnps = (flag & 0xFFFFu) | (nsnps << 16);
	out[slot] = r;
	if(bad)
		atomicOr(err, bad);
}


// ---------------------------------------------------------------------------------------------------
// FASTA text -> records (SeqIORead_fasta<S>::next_seq, SeqIORead_fasta.h:51-103, with SeqIORead<S>::getline(true), SeqIORead.h:85-121)
//   every line is trimmed of white space on both ends (:88-96); blank lines are skipped (getline(true)); a line whose first character is '>'
//   opens a record, its id is the text up to the first white space (:57-76); every other line is appended to the sequence of the open
//   record, interior white space included (:97).
// ---------------------------------------------------------------------------------------------------
constexpr int FA_ERR_NO_HEADER = 1, FA_ERR_EMPTY_ID = 2;

// one thread per line: trimmed extent and kind (0 blank, 1 header, 2 sequence)
__global__ void k_fa_classify(const char* __restrict__ text, uint64_t nbytes, const uint64_t* __restrict__ line_start, uint64_t nlines, uint64_t* __restrict__ line_a,
                              uint32_t* __restrict__ line_len, uint32_t* __restrict__ is_header, uint32_t* __restrict__ id_len, int* __restrict__ err)
{
	abw_grid_wait();
	const uint64_t l = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if(l >= nlines)
		return;
	auto [a, b] = line_extent(line_start, nlines, nbytes, l);
	while(a < b && dev_isspace(text[a]))
		a++;
	while(b > a && dev_isspace(text[b - 1]))
		b--;
	uint32_t hdr = 0, len = 0, idl = 0;
	if(b > a) {
		if(text[a] == '>') {
			hdr = 1;
			uint64_t q = a + 1;
			while(q < b && !dev_isspace(text[q]))
				q++;
			idl = (uint32_t)(q - (a + 1));
			if(idl == 0)
				atomicOr(err, FA_ERR_EMPTY_ID);          // "Was expeecting a header line ..." (:58-62)
		}
		else
			len = (uint32_t)min((uint64_t)0xFFFFFFFFu, b - a);
	}
	line_a[l] = a;
	line_len[l] = len;
	is_header[l] = hdr;
	id_len[l] = idl;
}

// per line: its record (headers seen so far - 1); header lines publish where the record starts in the running sum of sequence characters, and
// their description: the header after the id and the white space that follows it, up to the trimmed end of the line (SeqIORead_fasta.h:57-76)
__global__ void k_fa_records(const char* __restrict__ text, uint64_t nbytes, const uint64_t* __restrict__ line_start, const uint64_t* __restrict__ line_a,
                             const uint32_t* __restrict__ line_len, const uint32_t* __restrict__ is_header, const uint32_t* __restrict__ id_len,
                             const uint64_t* __restrict__ hdr_before, const uint64_t* __restrict__ chars_before, uint64_t nlines, uint64_t nrec,
                             uint64_t* __restrict__ rec_id_off, uint32_t* __restrict__ rec_id_len, uint64_t* __restrict__ rec_chars0,
                             uint64_t* __restrict__ rec_desc_off, uint32_t* __restrict__ rec_desc_len, int* __restrict__ err)
{
	abw_grid_wait();
	const uint64_t l = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if(l >= nlines)
		return;
	if(is_header[l]) {
		const uint64_t r = hdr_before[l];
		rec_id_off[r] = line_a[l] + 1;
		rec_id_len[r] = id_len[l];
		rec_chars0[r] = chars_before[l];
		uint64_t b = line_extent(line_start, nlines, nbytes, l).b, q = line_a[l] + 1 + id_len[l];
		while(b > q && dev_isspace(text[b - 1]))
			b--;
		while(q < b && dev_isspace(text[q]))
			q++;
		rec_desc_off[r] = q;
		rec_desc_len[r] = (uint32_t)min((uint64_t)0xFFFFFFFFu, b - q);
	}
	else if(line_len[l] && hdr_before[l] == 0)
		atomicOr(err, FA_ERR_NO_HEADER);                  // sequence text before the first header line (:58-62)
}

// one warp per sequence line: copy its trimmed text to where the record goes in the requested order
__global__ void __launch_bounds__(256) k_fa_copy(const char* __restrict__ text, const uint64_t* __restrict__ line_a, const uint32_t* __restrict__ line_len,
                                                 const uint64_t* __restrict__ hdr_before, const uint64_t* __restrict__ chars_before, uint64_t nlines,
                                                 const uint64_t* __restrict__ rec_chars0, const uint64_t* __restrict__ rec_dst, char* __restrict__ out)
{
	abw_grid_wait();
	const int lane = threadIdx.x & 31;
	const uint64_t warp0 = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
	for(uint64_t l = warp0; l < nlines; l += nwarps) {
		const uint32_t len = line_len[l];
		if(len == 0)
			continue;
		const uint64_t r = hdr_before[l] - 1;
		const uint64_t dst0 = rec_dst[r];
		if(dst0 == ~0ull)
			continue;                                       // record not wanted (e.g. a later record with a name already seen)
		const char* __restrict__ src = text + line_a[l];
		char* __restrict__ dst = out + dst0 + (chars_before[l] - rec_chars0[r]);
		for(uint32_t i = lane; i < len; i += 32)
			dst[i] = src[i];
	}
}


// one warp per sequence line: N (either case) and C/G (either case) of its characters, added to its record's counts
__global__ void __launch_bounds__(256) k_fa_base_counts(const char* __restrict__ text, const uint64_t* __restrict__ line_a, const uint32_t* __restrict__ line_len,
                                                        const uint64_t* __restrict__ hdr_before, uint64_t nlines, unsigned long long* __restrict__ countN,
                                                        unsigned long long* __restrict__ countGC)
{
	abw_grid_wait();
	const int lane = threadIdx.x & 31;
	const uint64_t warp0 = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
	for(uint64_t l = warp0; l < nlines; l += nwarps) {
		const uint32_t len = line_len[l];
		if(len == 0)
			continue;
		const char* __restrict__ src = text + line_a[l];
		uint32_t nN = 0, nGC = 0;
		for(uint32_t i = lane; i < len; i += 32) {
			const uint32_t c = (unsigned char)src[i] | 0x20u;            // 'N' and 'n' -> 'n', 'C' / 'c' -> 'c', 'G' / 'g' -> 'g'; no other byte maps there
			nN += c == 'n';
			nGC += c == 'c' || c == 'g';
		}
		nN = __reduce_add_sync(0xffffffffu, nN);
		nGC = __reduce_add_sync(0xffffffffu, nGC);
		if(lane == 0) {
			const uint64_t r = hdr_before[l] - 1;
			if(nN)
				atomicAdd(countN + r, (unsigned long long)nN);
			if(nGC)
				atomicAdd(countGC + r, (unsigned long long)nGC);
		}
	}
}

// ---------------------------------------------------------------------------------------------------
// .lrn data lines -> keys and a row-major matrix of doubles (ClusterData::ClusterData, ClusterData.cpp:110-168: one line per datapoint,
// "<key>\t<v1>\t...\t<vD>", values read with atof (:159); lines that are empty or start with '%' are skipped)
// ---------------------------------------------------------------------------------------------------
constexpr int LRN_ERR_FIELDS = 1;

__device__ double g_pow10[23] = {1e0, 1e1, 1e2, 1e3, 1e4, 1e5, 1e6, 1e7, 1e8, 1e9, 1e10, 1e11, 1e12, 1e13, 1e14, 1e15, 1e16, 1e17, 1e18, 1e19, 1e20, 1e21, 1e22};

// atof of the field [p, e).  Decimal numbers whose digits form an integer below 2^53 and whose decimal exponent is within +-22 are converted with ONE
// correctly rounded operation on two exactly representable doubles (the classic fast path of strtod), which is the correctly rounded result strtod
// returns; everything else (more digits, large exponents, "inf", "nan", hexadecimal) is left to the host: *exact = false.
__device__ __forceinline__ double dev_atof(const char* __restrict__ p, const char* __restrict__ e, bool* exact)
{
	*exact = true;
	while(p < e && dev_isspace(*p))
		p++;
	bool neg = false;
	if(p < e && (*p == '+' || *p == '-')) {
		neg = *p == '-';
		p++;
	}
	if(p < e && ((*p | 0x20) == 'i' || (*p | 0x20) == 'n')) {       // inf / nan
		*exact = false;
		return 0.0;
	}
	if(p + 1 < e && p[0] == '0' && (p[1] | 0x20) == 'x') {          // hexadecimal floating point
		*exact = false;
		return 0.0;
	}
	unsigned long long m = 0;
	int ndig = 0, frac = 0, sig = 0;
	bool any = false;
	while(p < e && *p >= '0' && *p <= '9') {
		if(sig > 0 || *p != '0') {
			if(sig < 19) m = m * 10 + (unsigned long long)(*p - '0');
			sig++;
		}
		any = true; ndig++; p++;
	}
	if(p < e && *p == '.') {
		p++;
		while(p < e && *p >= '0' && *p <= '9') {
			if(sig > 0 || *p != '0') {
				if(sig < 19) m = m * 10 + (unsigned long long)(*p - '0');
				sig++;
			}
			frac++;
			any = true; p++;
		}
	}
	if(!any)
		return 0.0;                                                // no conversion: atof returns 0
	int ex = 0;
	if(p < e && (*p | 0x20) == 'e') {
		const char* q = p + 1;
		bool eneg = false;
		if(q < e && (*q == '+' || *q == '-')) {
			eneg = *q == '-';
			q++;
		}
		if(q < e && *q >= '0' && *q <= '9') {
			int v = 0;
			while(q < e && *q >= '0' && *q <= '9') {
				if(v < 100000) v = v * 10 + (*q - '0');
				q++;
			}
			ex = eneg? -v : v;
		}
	}
	const int e10 = ex - frac;
	if(m == 0)
		return neg? -0.0 : 0.0;
	if(sig > 19 || m >= (1ull << 53) || e10 < -22 || e10 > 22) {
		*exact = false;
		return 0.0;
	}
	const double md = (double)m;                                  // exact
	const double r = (e10 >= 0)? __dmul_rn(md, g_pow10[e10]) : __ddiv_rn(md, g_pow10[-e10]);
	return neg? -r : r;
}

struct LrnFallback { uint64_t row; uint32_t col; uint32_t len; uint64_t off; };

__global__ void __launch_bounds__(128) k_lrn_parse(const char* __restrict__ text, uint64_t nbytes, const uint64_t* __restrict__ line_start, uint64_t nlines,
                                                   const uint32_t* __restrict__ is_row, const uint64_t* __restrict__ row_slot, uint32_t D, uint64_t cap,
                                                   uint64_t* __restrict__ keys, double* __restrict__ values, LrnFallback* __restrict__ fb, uint32_t fb_cap,
                                                   uint32_t* __restrict__ fb_count, int* __restrict__ err)
{
	abw_grid_wait();
	const uint64_t l = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if(l >= nlines || !is_row[l])
		return;
	const uint64_t row = row_slot[l];
	if(row >= cap)
		return;
	const auto [a, b] = line_extent(line_start, nlines, nbytes, l);
	const char* p = text + a;
	const char* e = text + b;
	while(e > p && dev_isspace(e[-1]))
		e--;
	uint32_t field = 0;
	const char* fs = p;
	for(const char* q = p;; q++) {
		if(q == e || *q == '\t') {
			if(field == 0)
				keys[row] = (uint64_t)(unsigned long)dev_atoi(fs, q);          // atoi of the key, ClusterData.cpp:151
			else if(field <= D) {
				bool exact;
				const double v = dev_atof(fs, q, &exact);
				values[row * D + (field - 1)] = v;
				if(!exact) {
					const uint32_t k = atomicAdd(fb_count, 1u);
					if(k < fb_cap) {
						fb[k].row = row; fb[k].col = field - 1; fb[k].len = (uint32_t)(q - fs); fb[k].off = (uint64_t)(fs - text);
					}
				}
			}
			field++;
			fs = q + 1;
			if(q == e)
				break;
		}
	}
	if(field != D + 1)
		atomicOr(err, LRN_ERR_FIELDS);                       // "number of dimensions found is ...", ClusterData.cpp:137-141
}

// one warp per destination row: dst[i][0 .. ncols) = src[rows[i]][0 .. ncols)
__global__ void __launch_bounds__(256) k_gather_rows(const double* __restrict__ src, uint64_t ld_src, double* __restrict__ dst, uint64_t ld_dst, uint32_t ncols,
                                                     const uint64_t* __restrict__ rows, uint64_t nrows)
{
	abw_grid_wait();
	const int lane = threadIdx.x & 31;
	const uint64_t nwarps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
	for(uint64_t i = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; i < nrows; i += nwarps) {
		const double* __restrict__ s = src + rows[i] * ld_src;
		double* __restrict__ d = dst + i * ld_dst;
		for(uint32_t c = lane; c < ncols; c += 32)
			d[c] = s[c];
	}
}

}  // namespace

struct abw_fasta {
	LineIndex lines;                          // the text; its line starts are released once the records are found
	uint64_t nrec = 0;
	DevBuf<uint64_t> line_a, hdr_before, chars_before, rec_id_off, rec_chars0, rec_desc_off;
	DevBuf<uint32_t> line_len, rec_id_len, rec_desc_len;
	// per record: sequence length, and what abw_fasta_format lays the text out with (id, description, first sequence character)
	std::vector<uint64_t> h_seq_len, h_id_off, h_desc_off, h_chars0;
	std::vector<uint32_t> h_id_len, h_desc_len;
};

extern "C" {

int abw_names_create(abw_ctx* ctx, const char* names_blob, const uint64_t* h_name_off, uint32_t nscaf, abw_names** out)
{
	if(!ctx || !out || !h_name_off || (!names_blob && nscaf && h_name_off[nscaf] > 0))
		return abw_fail(ctx, ABW_ERR_ARG, "abw_names_create: null argument");
	ABW_ENTER(ctx);
	abw_names* nm = new abw_names();
	int rc = [&]() -> int {
		nm->nscaf = nscaf;
		uint32_t nslots = 16;
		while(nslots < 2ull * nscaf + 1)
			nslots <<= 1;
		nm->nslots = nslots;
		std::vector<unsigned long long> sh(nslots, 0);
		std::vector<uint32_t> si(nslots, 0);
		for(uint32_t i = 0; i < nscaf; i++) {
			if(h_name_off[i + 1] < h_name_off[i])
				return abw_fail(ctx, ABW_ERR_ARG, "abw_names_create: offsets must be non-decreasing");
			const unsigned long long h = abw_fnv1a(names_blob + h_name_off[i], h_name_off[i + 1] - h_name_off[i]);
			uint32_t s = (uint32_t)(h & (nslots - 1));
			while(sh[s] != 0)
				s = (s + 1) & (nslots - 1);
			sh[s] = h;
			si[s] = i;
		}
		const uint64_t blob_bytes = h_name_off[nscaf];
		ABW_CUDA(ctx, nm->slot_hash.alloc(nslots));
		ABW_CUDA(ctx, nm->slot_index.alloc(nslots));
		ABW_CUDA(ctx, nm->blob.alloc(blob_bytes + 1));
		ABW_CUDA(ctx, nm->off.alloc((size_t)nscaf + 1));
		ABW_CUDA(ctx, cudaMemcpyAsync(nm->slot_hash.p, sh.data(), sizeof(unsigned long long) * nslots, cudaMemcpyHostToDevice, ctx->stream));
		ABW_CUDA(ctx, cudaMemcpyAsync(nm->slot_index.p, si.data(), sizeof(uint32_t) * nslots, cudaMemcpyHostToDevice, ctx->stream));
		if(blob_bytes)
			ABW_CUDA(ctx, cudaMemcpyAsync(nm->blob.p, names_blob, blob_bytes, cudaMemcpyHostToDevice, ctx->stream));
		ABW_CUDA(ctx, cudaMemcpyAsync(nm->off.p, h_name_off, sizeof(uint64_t) * ((size_t)nscaf + 1), cudaMemcpyHostToDevice, ctx->stream));
		ABW_CUDA(ctx, abw_sync(ctx));
		return ABW_OK;
	}();
	if(rc != ABW_OK) {
		delete nm;
		return rc;
	}
	*out = nm;
	return ABW_OK;
}

void abw_names_destroy(abw_names* n) { delete n; }

int abw_parse_sam(abw_ctx* ctx, const abw_names* names, const char* text, uint64_t nbytes, int text_on_device, abw_read* d_reads, uint64_t cap, uint64_t* nreads)
{
	if(!ctx || !names || !nreads || (!text && nbytes) || (!d_reads && cap))
		return abw_fail(ctx, ABW_ERR_ARG, "abw_parse_sam: null argument");
	ABW_ENTER(ctx);
	*nreads = 0;
	if(nbytes == 0)
		return ABW_OK;
	DevBuf<int> d_err;
	ABW_CUDA(ctx, d_err.alloc(1));
	ABW_CUDA(ctx, cudaMemsetAsync(d_err.p, 0, sizeof(int), ctx->stream));
	LineIndex li;
	ABW_CHECK(line_index(ctx, text, nbytes, text_on_device, &li));
	DevBuf<uint32_t> is_record;
	DevBuf<uint64_t> rec_slot;
	uint64_t nrec = 0;
	ABW_CHECK(select_lines(ctx, li, '@', false, is_record, rec_slot, &nrec));
	*nreads = nrec;
	if(nrec > cap)
		return abw_fail(ctx, ABW_ERR_ARG, "abw_parse_sam: the record buffer is too small for this chunk (nreads holds the number needed)");
	if(nrec) {
		ABW_LAUNCH(ctx, k_sam_parse, abw_div_up(li.nlines, 128), 128, 0, li.text, nbytes, li.start.p, li.nlines, is_record.p, rec_slot.p, names->slot_hash.p,
		           names->slot_index.p, names->nslots, names->blob.p, names->off.p, d_reads, cap, d_err.p);
	}
	int h_err = 0;
	ABW_CUDA(ctx, abw_fetch(ctx, &h_err, d_err.p, sizeof(int)));
	ABW_CUDA(ctx, abw_sync(ctx));
	if(h_err & SAM_ERR_LOWER_N)
		return abw_fail(ctx, ABW_ERR_ILLEGAL_DNA, "Illegal_DNAString: lower-case 'n' in a read sequence (String.cpp:47-49)");
	if(h_err & SAM_ERR_FEW_FIELDS)
		return abw_fail(ctx, ABW_ERR_ARG, "abw_parse_sam: a SAM line has fewer than 11 tab-separated fields (ReadMapping.cpp:36-51 reads fs[10])");
	if(h_err & SAM_ERR_MDZ)
		return abw_fail(ctx, ABW_ERR_ARG, "abw_parse_sam: Illegal SNPs description in an MD:Z field (Illegal_mapping, ReadMapping.cpp:100-113)");
	return ABW_OK;
}

int abw_fasta_scan(abw_ctx* ctx, const char* text, uint64_t nbytes, int text_on_device, abw_fasta** out)
{
	if(!ctx || !out || (!text && nbytes))
		return abw_fail(ctx, ABW_ERR_ARG, "abw_fasta_scan: null argument");
	ABW_ENTER(ctx);
	abw_fasta* f = new abw_fasta();
	int rc = [&]() -> int {
		if(nbytes == 0)
			return ABW_OK;
		DevBuf<uint32_t> is_header, id_len;
		DevBuf<uint64_t> total;
		DevBuf<int> d_err;
		ABW_CUDA(ctx, total.alloc(2));
		ABW_CUDA(ctx, d_err.alloc(1));
		ABW_CUDA(ctx, cudaMemsetAsync(d_err.p, 0, sizeof(int), ctx->stream));
		LineIndex& li = f->lines;
		ABW_CHECK(line_index(ctx, text, nbytes, text_on_device, &li));
		const uint64_t nlines = li.nlines;
		ABW_CUDA(ctx, f->line_a.alloc(nlines));
		ABW_CUDA(ctx, f->line_len.alloc(nlines));
		ABW_CUDA(ctx, is_header.alloc(nlines));
		ABW_CUDA(ctx, id_len.alloc(nlines));
		ABW_CUDA(ctx, f->hdr_before.alloc(nlines));
		ABW_CUDA(ctx, f->chars_before.alloc(nlines));
		ABW_LAUNCH(ctx, k_fa_classify, abw_div_up(nlines, 256), 256, 0, li.text, nbytes, li.start.p, nlines, f->line_a.p, f->line_len.p, is_header.p, id_len.p, d_err.p);
		// hdr_before[l] = header lines strictly before l; a header line itself gets its own record index, a sequence line index + 1 of its record
		ABW_CHECK(abw_exclusive_scan_u32_to_u64(ctx, is_header.p, f->hdr_before.p, nlines, total.p));
		ABW_CHECK(abw_exclusive_scan_u32_to_u64(ctx, f->line_len.p, f->chars_before.p, nlines, total.p + 1));
		uint64_t tot[2] = {0, 0};
		ABW_CUDA(ctx, abw_fetch(ctx, tot, total.p, 2 * sizeof(uint64_t)));
		ABW_CUDA(ctx, abw_sync(ctx));
		const uint64_t nrec = tot[0], nchars = tot[1];
		f->nrec = nrec;
		ABW_CUDA(ctx, f->rec_id_off.alloc(nrec));
		ABW_CUDA(ctx, f->rec_id_len.alloc(nrec));
		ABW_CUDA(ctx, f->rec_chars0.alloc(nrec + 1));
		ABW_CUDA(ctx, f->rec_desc_off.alloc(nrec));
		ABW_CUDA(ctx, f->rec_desc_len.alloc(nrec));
		ABW_LAUNCH(ctx, k_fa_records, abw_div_up(nlines, 256), 256, 0, li.text, nbytes, li.start.p, f->line_a.p, f->line_len.p, is_header.p, id_len.p, f->hdr_before.p,
		           f->chars_before.p, nlines, nrec, f->rec_id_off.p, f->rec_id_len.p, f->rec_chars0.p, f->rec_desc_off.p, f->rec_desc_len.p, d_err.p);
		li.start.release();
		ABW_CUDA(ctx, cudaMemcpyAsync(f->rec_chars0.p + nrec, &nchars, sizeof(uint64_t), cudaMemcpyHostToDevice, ctx->stream));
		int h_err = 0;
		ABW_CUDA(ctx, abw_fetch(ctx, &h_err, d_err.p, sizeof(int)));
		f->h_chars0.resize(nrec + 1);
		f->h_id_off.resize(nrec);
		f->h_id_len.resize(nrec);
		f->h_desc_off.resize(nrec);
		f->h_desc_len.resize(nrec);
		ABW_CUDA(ctx, abw_fetch(ctx, f->h_chars0.data(), f->rec_chars0.p, sizeof(uint64_t) * (nrec + 1)));
		if(nrec) {
			ABW_CUDA(ctx, abw_fetch(ctx, f->h_id_off.data(), f->rec_id_off.p, sizeof(uint64_t) * nrec));
			ABW_CUDA(ctx, abw_fetch(ctx, f->h_id_len.data(), f->rec_id_len.p, sizeof(uint32_t) * nrec));
			ABW_CUDA(ctx, abw_fetch(ctx, f->h_desc_off.data(), f->rec_desc_off.p, sizeof(uint64_t) * nrec));
			ABW_CUDA(ctx, abw_fetch(ctx, f->h_desc_len.data(), f->rec_desc_len.p, sizeof(uint32_t) * nrec));
		}
		ABW_CUDA(ctx, abw_sync(ctx));
		if(h_err)
			return abw_fail(ctx, ABW_ERR_ARG, "Bad_file: was expecting a header line for the next sequence in a fasta file but got something else (SeqIORead_fasta.h:58-62)");
		f->h_seq_len.resize(nrec);
		for(uint64_t r = 0; r < nrec; r++)
			f->h_seq_len[r] = f->h_chars0[r + 1] - f->h_chars0[r];
		// from here on a sequence line looks its record up as hdr_before - 1
		return ABW_OK;
	}();
	if(rc != ABW_OK) {
		delete f;
		return rc;
	}
	*out = f;
	return ABW_OK;
}

void abw_fasta_destroy(abw_fasta* f) { delete f; }

uint64_t abw_fasta_count(const abw_fasta* f) { return f? f->nrec : 0; }

int abw_fasta_get(abw_ctx* ctx, const abw_fasta* f, uint64_t* h_id_off, uint32_t* h_id_len, uint64_t* h_seq_len)
{
	if(!ctx || !f)
		return abw_fail(ctx, ABW_ERR_ARG, "abw_fasta_get: null argument");
	if(f->nrec == 0)
		return ABW_OK;
	if(h_id_off)
		ABW_CUDA(ctx, abw_fetch(ctx, h_id_off, f->rec_id_off.p, sizeof(uint64_t) * f->nrec));
	if(h_id_len)
		ABW_CUDA(ctx, abw_fetch(ctx, h_id_len, f->rec_id_len.p, sizeof(uint32_t) * f->nrec));
	ABW_CUDA(ctx, abw_sync(ctx));
	if(h_seq_len)
		memcpy(h_seq_len, f->h_seq_len.data(), sizeof(uint64_t) * f->nrec);
	return ABW_OK;
}

int abw_fasta_pack(abw_ctx* ctx, const abw_fasta* f, const uint32_t* h_order, uint32_t nout, abw_seqset** out)
{
	if(!ctx || !f || !out || (!h_order && nout))
		return abw_fail(ctx, ABW_ERR_ARG, "abw_fasta_pack: null argument");
	ABW_ENTER(ctx);
	std::vector<uint64_t> offsets((size_t)nout + 1, 0), rec_dst(f->nrec, ~0ull);
	for(uint32_t i = 0; i < nout; i++) {
		if(h_order[i] >= f->nrec)
			return abw_fail(ctx, ABW_ERR_ARG, "abw_fasta_pack: record index out of range");
		if(rec_dst[h_order[i]] != ~0ull)
			return abw_fail(ctx, ABW_ERR_ARG, "abw_fasta_pack: a record may appear only once in the order");
		rec_dst[h_order[i]] = offsets[i];
		offsets[i + 1] = offsets[i] + f->h_seq_len[h_order[i]];
	}
	DevBuf<char> ascii;
	DevBuf<uint64_t> d_dst;
	ABW_CUDA(ctx, ascii.alloc(offsets[nout] + 64));
	ABW_CUDA(ctx, d_dst.alloc(f->nrec));
	if(f->nrec) {
		ABW_CUDA(ctx, cudaMemcpyAsync(d_dst.p, rec_dst.data(), sizeof(uint64_t) * f->nrec, cudaMemcpyHostToDevice, ctx->stream));
		const unsigned int blocks = (unsigned int)std::min<uint64_t>(abw_div_up(f->lines.nlines * 32, 256), (uint64_t)ctx->sm_count * 16);
		ABW_LAUNCH(ctx, k_fa_copy, blocks, 256, 0, f->lines.text, f->line_a.p, f->line_len.p, f->hdr_before.p, f->chars_before.p, f->lines.nlines, f->rec_chars0.p, d_dst.p,
		           ascii.p);
	}
	ABW_CUDA(ctx, abw_sync(ctx));      // rec_dst is a local
	return abw_pack_sequences(ctx, ascii.p, 1, offsets.data(), nout, out);
}

int abw_fasta_format(abw_ctx* ctx, const abw_fasta* f, const uint32_t* h_recs, uint64_t nrecs, uint64_t byte0, char* d_text, uint64_t cap, uint64_t* total_bytes,
                     uint64_t* nbytes)
{
	if(!ctx || !f || !total_bytes || !nbytes || (!h_recs && nrecs))
		return abw_fail(ctx, ABW_ERR_ARG, "abw_fasta_format: null argument");
	ABW_ENTER(ctx);
	*total_bytes = 0;
	*nbytes = 0;
	std::vector<FaRecord> recs(nrecs);
	for(uint64_t i = 0; i < nrecs; i++) {
		const uint32_t r = h_recs[i];
		if(r >= f->nrec)
			return abw_fail(ctx, ABW_ERR_ARG, "abw_fasta_format: record index out of range");
		recs[i] = FaRecord{f->h_id_off[r], f->h_desc_off[r], f->h_chars0[r], f->h_seq_len[r], 0, 0, f->h_id_len[r], f->h_desc_len[r]};
	}
	FaSource src;
	src.kind = FA_SRC_TEXT;
	src.text = f->lines.text;
	src.line_a = f->line_a.p;
	src.line_len = f->line_len.p;
	src.chars_before = f->chars_before.p;
	src.nlines = f->lines.nlines;
	return abw_fasta_text(ctx, src, recs, byte0, d_text, cap, total_bytes, nbytes);
}

int abw_fasta_base_counts(abw_ctx* ctx, const abw_fasta* f, uint64_t* h_count_N, uint64_t* h_count_GC)
{
	if(!ctx || !f || ((!h_count_N || !h_count_GC) && f->nrec))
		return abw_fail(ctx, ABW_ERR_ARG, "abw_fasta_base_counts: null argument");
	ABW_ENTER(ctx);
	if(f->nrec == 0)
		return ABW_OK;
	DevBuf<unsigned long long> counts;
	ABW_CUDA(ctx, counts.alloc(2 * f->nrec));
	ABW_CUDA(ctx, cudaMemsetAsync(counts.p, 0, sizeof(unsigned long long) * 2 * f->nrec, ctx->stream));
	const unsigned int blocks = (unsigned int)std::min<uint64_t>(abw_div_up(f->lines.nlines * 32, 256), (uint64_t)ctx->sm_count * 16);
	ABW_LAUNCH(ctx, k_fa_base_counts, blocks, 256, 0, f->lines.text, f->line_a.p, f->line_len.p, f->hdr_before.p, f->lines.nlines, counts.p, counts.p + f->nrec);
	ABW_CUDA(ctx, abw_fetch(ctx, h_count_N, counts.p, sizeof(uint64_t) * f->nrec));
	ABW_CUDA(ctx, abw_fetch(ctx, h_count_GC, counts.p + f->nrec, sizeof(uint64_t) * f->nrec));
	ABW_CUDA(ctx, abw_sync(ctx));
	return ABW_OK;
}

int abw_parse_lrn(abw_ctx* ctx, const char* text, uint64_t nbytes, int text_on_device, uint32_t D, uint64_t* d_keys, double* d_values, uint64_t cap_rows, uint64_t* nrows)
{
	if(!ctx || !nrows || (!text && nbytes) || D == 0 || ((!d_keys || !d_values) && cap_rows))
		return abw_fail(ctx, ABW_ERR_ARG, "abw_parse_lrn: bad argument");
	ABW_ENTER(ctx);
	*nrows = 0;
	if(nbytes == 0)
		return ABW_OK;
	DevBuf<uint32_t> fb_count;
	DevBuf<LrnFallback> fb;
	DevBuf<int> d_err;
	const uint32_t fb_cap = 1u << 20;
	ABW_CUDA(ctx, d_err.alloc(1));
	ABW_CUDA(ctx, fb_count.alloc(1));
	ABW_CUDA(ctx, fb.alloc(fb_cap));
	ABW_CUDA(ctx, cudaMemsetAsync(d_err.p, 0, sizeof(int), ctx->stream));
	ABW_CUDA(ctx, cudaMemsetAsync(fb_count.p, 0, sizeof(uint32_t), ctx->stream));
	LineIndex li;
	ABW_CHECK(line_index(ctx, text, nbytes, text_on_device, &li));
	DevBuf<uint32_t> is_row;
	DevBuf<uint64_t> row_slot;
	uint64_t nr = 0;
	ABW_CHECK(select_lines(ctx, li, '%', true, is_row, row_slot, &nr));
	*nrows = nr;
	if(nr > cap_rows)
		return abw_fail(ctx, ABW_ERR_ARG, "abw_parse_lrn: more data lines than the caller made room for (nrows holds the number found)");
	if(nr == 0)
		return ABW_OK;
	ABW_LAUNCH(ctx, k_lrn_parse, abw_div_up(li.nlines, 128), 128, 0, li.text, nbytes, li.start.p, li.nlines, is_row.p, row_slot.p, D, cap_rows, d_keys, d_values, fb.p,
	           fb_cap, fb_count.p, d_err.p);
	int h_err = 0;
	uint32_t h_fb = 0;
	ABW_CUDA(ctx, abw_fetch(ctx, &h_err, d_err.p, sizeof(int)));
	ABW_CUDA(ctx, abw_fetch(ctx, &h_fb, fb_count.p, sizeof(uint32_t)));
	ABW_CUDA(ctx, abw_sync(ctx));
	if(h_err & LRN_ERR_FIELDS)
		return abw_fail(ctx, ABW_ERR_ARG, "abw_parse_lrn: a data line does not have the expected number of tab-separated fields (ClusterData.cpp:137-141)");
	if(h_fb > fb_cap)
		return abw_fail(ctx, ABW_ERR_UNSUPPORTED, "abw_parse_lrn: too many values outside the exact decimal fast path");
	if(h_fb > 0) {
		// values that need full strtod (more than 19 digits, exponents beyond +-22, inf/nan, hexadecimal): converted on the host with the C library, as atof does
		std::vector<LrnFallback> h(h_fb);
		ABW_CUDA(ctx, abw_fetch(ctx, h.data(), fb.p, sizeof(LrnFallback) * h_fb));
		ABW_CUDA(ctx, abw_sync(ctx));
		std::vector<char> tmp;
		for(const LrnFallback& f : h) {
			tmp.assign((size_t)f.len + 1, 0);
			if(text_on_device)
				ABW_CUDA(ctx, cudaMemcpy(tmp.data(), li.text + f.off, f.len, cudaMemcpyDeviceToHost));
			else
				memcpy(tmp.data(), text + f.off, f.len);
			const double v = atof(tmp.data());
			ABW_CUDA(ctx, cudaMemcpyAsync(d_values + f.row * D + f.col, &v, sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
			ABW_CUDA(ctx, abw_sync(ctx));
		}
	}
	return ABW_OK;
}

int abw_gather_rows(abw_ctx* ctx, const double* d_src, uint64_t ld_src, const uint64_t* rows, int rows_on_device, uint64_t nrows, uint32_t ncols, double* d_dst,
                    uint64_t ld_dst)
{
	if(!ctx || (nrows && (!d_src || !d_dst || !rows)) || ld_dst < ncols)
		return abw_fail(ctx, ABW_ERR_ARG, "abw_gather_rows: bad argument");
	ABW_ENTER(ctx);
	if(nrows == 0 || ncols == 0)
		return ABW_OK;
	DevBuf<uint64_t> d_rows;
	const uint64_t* r = rows;
	if(!rows_on_device) {
		ABW_CUDA(ctx, d_rows.alloc(nrows));
		ABW_CUDA(ctx, cudaMemcpyAsync(d_rows.p, rows, nrows * sizeof(uint64_t), cudaMemcpyHostToDevice, ctx->stream));
		r = d_rows.p;
	}
	const unsigned int blocks = (unsigned int)std::min<uint64_t>(abw_div_up(nrows, 8), (uint64_t)ctx->sm_count * 16);
	ABW_LAUNCH(ctx, k_gather_rows, blocks, 256, 0, d_src, ld_src, d_dst, ld_dst, ncols, r, nrows);
	if(!rows_on_device)
		ABW_CUDA(ctx, abw_sync(ctx));      // the host row list may change once the call returns
	return ABW_OK;
}

}  // extern "C"
