// Host-side helpers shared by the two command-line programs (abawaca-build, abawaca) of abawaca_b200.
// Everything here is parsing and formatting at the on-disk boundary (SURVEY.md appendix A); all computation
// goes through the C ABI of libabawaca_b200.so.  Written from the format descriptions, not from the reference code.
#pragma once
#include <algorithm>
#include <chrono>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <cctype>
#include <map>
#include <stdexcept>
#include <string>
#include <vector>
#include <glob.h>
#include <sys/stat.h>
#include "../../include/abawaca_b200.h"

namespace abwh {

inline std::string read_file(const std::string& path)
{
	std::string text;
	FILE* fp = fopen(path.c_str(), "rb");
	if(!fp)
		throw std::runtime_error("Failed to open file " + path);
	fseek(fp, 0, SEEK_END);
	const long sz = ftell(fp);
	rewind(fp);
	text.resize((size_t)(sz > 0? sz : 0));
	if(sz > 0 && fread(&text[0], 1, (size_t)sz, fp) != (size_t)sz) {
		fclose(fp);
		throw std::runtime_error("Failed to read file " + path);
	}
	fclose(fp);
	return text;
}

// a UCSC .2bit file starts with the signature 0x1A412743 in the byte order of the file
inline bool is_twobit(const std::string& bytes)
{
	if(bytes.size() < 4)
		return false;
	const unsigned char* b = (const unsigned char*)bytes.data();
	return (b[0] == 0x43 && b[1] == 0x27 && b[2] == 0x41 && b[3] == 0x1A) || (b[0] == 0x1A && b[1] == 0x41 && b[2] == 0x27 && b[3] == 0x43);
}

// a BAM file starts with a BGZF block header (gzip magic 1f 8b); no SAM file starts with byte 0x1F.  Leaves the file at its start.
inline bool is_bgzf(FILE* fp)
{
	unsigned char b[2] = {0, 0};
	const size_t n = fread(b, 1, 2, fp);
	rewind(fp);
	return n == 2 && b[0] == 0x1F && b[1] == 0x8B;
}

inline bool directory_exists(const std::string& d)
{
	struct stat st;
	return stat(d.c_str(), &st) == 0 && S_ISDIR(st.st_mode);
}

inline bool file_readable(const std::string& f)
{
	FILE* fp = fopen(f.c_str(), "r");
	if(!fp)
		return false;
	fclose(fp);
	return true;
}

inline std::vector<std::string> glob_files(const std::string& pattern)
{
	glob_t g;
	std::vector<std::string> out;
	if(glob(pattern.c_str(), GLOB_TILDE, nullptr, &g) == 0)
		for(size_t i = 0; i < g.gl_pathc; i++)
			out.push_back(g.gl_pathv[i]);
	globfree(&g);
	return out;
}

#define ABWH_CHECK(ctx, call)                                                                           \
	do {                                                                                                \
		int rc__ = (call);                                                                              \
		if(rc__ != ABW_OK)                                                                              \
			throw std::runtime_error(std::string(#call) + " failed: " + abw_last_error(ctx));           \
	} while(0)

// ABW_TIMING=1: wall-clock milestones on stderr, each with the time since the one before (where the time of a command line goes)
inline void milestone(const std::string& what)
{
	static const bool on = getenv("ABW_TIMING") != nullptr;
	static auto t0 = std::chrono::steady_clock::now();
	if(!on)
		return;
	const auto t1 = std::chrono::steady_clock::now();
	fprintf(stderr, "[abw timing] %-28s %8.3f s\n", what.c_str(), std::chrono::duration<double>(t1 - t0).count());
	t0 = t1;
}

// the data lines of a .lrn file are made on the device (abw_format_lrn) in pieces of at most LRN_CHUNK bytes
const uint64_t LRN_CHUNK = (uint64_t)64 << 20;

// Writes a .lrn file (ClusterData.cpp:27-168 reads it back): the header "% <nlines>", "% <columns + 1>", "% 9" and "\t1" per column, "% Key" and
// the column names; then line i = "<r+1>" and the values of row r = rows[i] (r = i when rows is NULL; rows in host memory) of the row-major device
// matrix d_values (row stride ld), printed as fmt (ABW_TEXT_*).  d_text (LRN_CHUNK bytes of device memory) and text are scratch, kept from file to
// file.  false when fp takes fewer bytes than it is given.
inline bool write_lrn(abw_ctx* ctx, FILE* fp, const std::vector<std::string>& names, const double* d_values, uint64_t ld, const uint64_t* rows, uint64_t nlines,
                      int fmt, char* d_text, std::vector<char>& text)
{
	fprintf(fp, "%% %lu\n%% %lu\n%% 9", (unsigned long)nlines, (unsigned long)(names.size() + 1));
	for(size_t c = 0; c < names.size(); c++) fprintf(fp, "\t1");
	fprintf(fp, "\n%% Key");
	for(const std::string& n : names) fprintf(fp, "\t%s", n.c_str());
	fprintf(fp, "\n");
	for(uint64_t line0 = 0; line0 < nlines;) {
		uint64_t done = 0, nbytes = 0;
		ABWH_CHECK(ctx, abw_format_lrn(ctx, d_values, ld, 0, (uint32_t)names.size(), rows, 0, line0, nlines, fmt, d_text, LRN_CHUNK, &done, &nbytes));
		text.resize(std::max<size_t>(text.size(), nbytes));
		ABWH_CHECK(ctx, abw_copy_to_host(ctx, text.data(), d_text, nbytes));
		if(fwrite(text.data(), 1, nbytes, fp) != nbytes)
			return false;
		line0 += done;
	}
	return true;
}

}  // namespace abwh
