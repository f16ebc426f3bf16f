// The FASTA writer of fastaout.cu, shared by the FASTA (ingest.cu) and .2bit (seqcodec.cu) handles: each fills one FaRecord per record it is asked
// for and says where the bytes lie.
#pragma once
#include "common.cuh"

// One record of the output: its header is '>' + text[id_off, +id_len) + ' ' + text[desc_off, +desc_len) + '\n', its sequence `len` bases.
// FA_SRC_TEXT: base k is the (seq0 + k)-th character of the sequence lines of the FASTA text, counted over the whole file.
// FA_SRC_2BIT: base k is 'N' under N block [nb0, nb1) of the block table, else the 2-bit code at bit 6 - 2 (k & 3) of text[seq0 + k / 4] as TCAG.
struct FaRecord {
	uint64_t id_off, desc_off, seq0, len, nb0, nb1;
	uint32_t id_len, desc_len;
};

constexpr int FA_SRC_TEXT = 0, FA_SRC_2BIT = 1;

struct FaSource {
	int kind = FA_SRC_TEXT;
	const char* text = nullptr;              // FASTA text or .2bit image, device memory
	// FA_SRC_TEXT: the line table of abw_fasta_scan (trimmed start, sequence characters and sequence characters before, per line)
	const uint64_t* line_a = nullptr;
	const uint32_t* line_len = nullptr;
	const uint64_t* chars_before = nullptr;
	uint64_t nlines = 0;
	// FA_SRC_2BIT: N blocks {start, size} of all records
	const uint2* nblocks = nullptr;
};

// Bytes [byte0, byte0 + cap) of the text of the records `recs`, in list order, to d_text, as abw_fasta_format describes.  One wait on the context
// stream, at the end.
int abw_fasta_text(abw_ctx* ctx, const FaSource& src, const std::vector<FaRecord>& recs, uint64_t byte0, char* d_text, uint64_t cap, uint64_t* total,
                   uint64_t* nbytes);
