// Device-resident objects of the feature stage, shared by features.cu (pack, windows, k-mer signature) and coverage.cu.
#pragma once
#include "common.cuh"

struct abw_seqset {
	uint32_t nscaf = 0;
	uint64_t total_padded = 0;            // bases
	DevBuf<uint64_t> len, base;           // [nscaf], [nscaf+1]
	DevBuf<uint32_t> packed, valid, nmask;
	DevBuf<unsigned long long> countN, countGC;
	std::vector<uint64_t> h_len, h_base;
};

struct abw_segments {
	uint32_t nscaf = 0;
	uint64_t nseg = 0;
	DevBuf<uint64_t> seg_first;           // [nscaf+1]
	DevBuf<uint32_t> seg_scaf;            // [nseg]
	DevBuf<uint64_t> seg_start, seg_end, seg_nonN;   // 1-based inclusive, abawaca-build.cpp:216
	DevBuf<uint64_t> seg_gbase;           // absolute (padded) base index of the first base of the segment
	DevBuf<uint4> scaf_info;              // per scaffold {first window (low 32 bits), windows, non-N bases per window (u64)}: one load for the coverage kernels
};

// scaf_info.w of a scaffold whose windows are all nbps characters long (no N): coverage then needs no window table for its reads
constexpr uint32_t COV_REGULAR = 0x80000000u;

// readcodec.cu: enqueues the decode of an ABW_READS_SORTED sample (arrays checked by abw_coverage_batch) into d_out[sm.nreads] on the context stream
int abw_decode_sorted_reads(abw_ctx* ctx, const abw_sample& sm, abw_read8* d_out);
