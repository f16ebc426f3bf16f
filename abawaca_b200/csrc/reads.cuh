// Pieces of a read record that the SAM text parser (ingest.cu) and the BAM parser (bam.cu) share: the scaffold-name table and its probe,
// and the SNP count of an MD:Z description.
#pragma once
#include "common.cuh"

struct abw_names {
	uint32_t nscaf = 0, nslots = 0;
	DevBuf<unsigned long long> slot_hash;     // open addressing, 0 = empty (hashes are forced non-zero)
	DevBuf<uint32_t> slot_index;
	DevBuf<char> blob;                        // concatenated names
	DevBuf<uint64_t> off;                     // [nscaf+1]
};

__host__ __device__ __forceinline__ unsigned long long abw_fnv1a(const char* s, uint64_t n)
{
	unsigned long long h = 1469598103934665603ull;
	for(uint64_t i = 0; i < n; i++) {
		h ^= (unsigned char)s[i];
		h *= 1099511628211ull;
	}
	return h? h : 1ull;
}

// index of the name s[0 .. n) in the table, 0xFFFFFFFF if it is not there (scafs.find(ref_name), abawaca-build.cpp:549)
__device__ __forceinline__ uint32_t abw_name_probe(const char* s, uint64_t n, const unsigned long long* __restrict__ slot_hash, const uint32_t* __restrict__ slot_index,
                                                   uint32_t nslots, const char* __restrict__ name_blob, const uint64_t* __restrict__ name_off)
{
	const unsigned long long h = abw_fnv1a(s, n);
	uint32_t slot = (uint32_t)(h & (nslots - 1));
	for(uint32_t probe = 0; probe < nslots; probe++) {
		const unsigned long long sh = slot_hash[slot];
		if(sh == 0)
			break;
		if(sh == h) {
			const uint32_t idx = slot_index[slot];
			const uint64_t a = name_off[idx], b = name_off[idx + 1];
			bool same = (b - a) == n;
			for(uint64_t i = 0; same && i < n; i++)
				same = name_blob[a + i] == s[i];
			if(same)
				return idx;
		}
		slot = (slot + 1) & (nslots - 1);
	}
	return 0xFFFFFFFFu;
}

// The SNP letters of the MD:Z description [m, me) as ReadMapping::determine_snps walks it (ReadMapping.cpp:94-125): MD:Z:[0-9]+(([A-Z]|\^[^0-9]+)[0-9]+)*,
// one per mismatch letter and one per deleted reference base.  Adds them to *nsnps; false for a description that does not follow the pattern
// (Illegal_mapping, :100-113).
__device__ __forceinline__ bool abw_md_snps(const char* m, const char* me, uint32_t* nsnps)
{
	uint32_t n = *nsnps;
	bool ok = true;
	while(m < me && *m >= '0' && *m <= '9')
		m++;
	while(m < me) {
		if(*m == '^') {
			m++;
			while(m < me && !(*m >= '0' && *m <= '9')) {
				n++;
				m++;
			}
		}
		else if(*m >= 'A' && *m <= 'Z') {
			n++;
			m++;
		}
		else {
			ok = false;
			break;
		}
		if(m >= me || !(*m >= '0' && *m <= '9')) {
			ok = false;
			break;
		}
		while(m < me && *m >= '0' && *m <= '9')
			m++;
	}
	*nsnps = n;
	return ok;
}
