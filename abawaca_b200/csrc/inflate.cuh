// Raw DEFLATE (RFC 1951) decoding of one BGZF block, and the CRC-32 of gzip, for the device (bam.cu) and for the host (the CPU tests build
// this header with g++ and compare it against zlib).
//
// The decoder accepts exactly what zlib's inflate accepts for a raw stream that has to end inside the given input:
//  * BTYPE 3, a stored block whose NLEN is not the complement of LEN, more than 286 literal/length or 30 distance codes, a code-length repeat
//    with nothing to repeat or running past the code lengths, and a dynamic block without an end-of-block code are errors;
//  * a code set that is over-subscribed is an error; one that is incomplete is an error too, except a literal/length or distance code with a
//    single code of length 1 (zlib allows that one; a distance code may also be empty, and using an unassigned code is then an error);
//  * literal/length symbols 286-287 and distance symbols 30-31 (reachable through the fixed code) are errors, as is a distance before the
//    first byte of the output;
//  * reading past the end of the input is an error; so is output past `cap` (a BGZF block's ISIZE).
// Codes are decoded through a table indexed by the next FAST bits of the stream; longer codes take the canonical walk of the counts.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define ABW_HD __host__ __device__ __forceinline__
#else
#define ABW_HD inline
#endif

namespace abw_inflate {

constexpr int LFAST = 10, DFAST = 8;      // first-level bits of the literal/length and distance tables

enum {
	OK = 0,
	E_BTYPE = 1,       // block type 3
	E_STORED = 2,      // stored block: LEN and NLEN disagree
	E_HEADER = 3,      // dynamic block header: too many codes, bad repeat, missing end-of-block code
	E_CODES = 4,       // over-subscribed or incomplete code set
	E_SYMBOL = 5,      // a bit pattern without a code, or symbol 286/287 or distance 30/31
	E_DIST = 6,        // distance before the first output byte
	E_OUTPUT = 7,      // output past cap
	E_INPUT = 8,       // input past the end
};

// 3.6 KB: what one decoder needs besides the input and output (in shared memory on the device)
struct Tables {
	uint16_t lcount[16], dcount[16];
	uint16_t lsym[288], dsym[32];
	uint16_t lfast[1 << LFAST], dfast[1 << DFAST];
	uint8_t  lens[320];
};

// LSB-first bit reader with a 64-bit buffer; bytes past the end read as 0 and are caught by overrun()
struct Bits {
	const uint8_t* in;
	uint32_t n, pos;
	int cnt;
	uint64_t buf;
	ABW_HD void refill()
	{
		while(cnt <= 56) {
			const uint64_t b = (pos < n)? in[pos] : 0u;
			pos++;
			buf |= b << cnt;
			cnt += 8;
		}
	}
	ABW_HD uint32_t take(int k)         // k <= cnt
	{
		const uint32_t v = (uint32_t)(buf & ((1ull << k) - 1));
		buf >>= k;
		cnt -= k;
		return v;
	}
	ABW_HD bool overrun() const { return (uint64_t)pos * 8 - (uint64_t)cnt > (uint64_t)n * 8; }
};

// Canonical code from code lengths: counts per length, symbols in code order, and the first-level table (entry = symbol << 4 | length, 0 = longer
// code).  kind 0: the code-length code (must be complete); 1: literal/length or distance code (a single code of length 1, or none, is allowed).
ABW_HD int build(const uint8_t* lens, int n, int kind, uint16_t* count, uint16_t* symbol, uint16_t* fast, int fb)
{
	uint16_t offs[16];
	for(int l = 0; l < 16; l++)
		count[l] = 0;
	for(int s = 0; s < n; s++)
		count[lens[s]]++;
	int left = 1, max = 0;
	for(int l = 1; l < 16; l++) {
		left <<= 1;
		left -= count[l];
		if(left < 0)
			return E_CODES;
		if(count[l])
			max = l;
	}
	if(left > 0 && (kind == 0 || max > 1))
		return E_CODES;
	offs[1] = 0;
	for(int l = 1; l < 15; l++)
		offs[l + 1] = offs[l] + count[l];
	for(int s = 0; s < n; s++)
		if(lens[s])
			symbol[offs[lens[s]]++] = (uint16_t)s;
	for(int i = 0; i < (1 << fb); i++)
		fast[i] = 0;
	uint32_t code = 0;
	int idx = 0;
	for(int l = 1; l <= fb; l++) {
		for(int j = 0; j < count[l]; j++, code++) {
			uint32_t rev = 0;
			for(int b = 0; b < l; b++)
				rev |= ((code >> b) & 1u) << (l - 1 - b);
			const uint16_t e = (uint16_t)((symbol[idx++] << 4) | l);
			for(uint32_t k = rev; k < (1u << fb); k += 1u << l)
				fast[k] = e;
		}
		code <<= 1;
	}
	return OK;
}

// next symbol, or -1 for a bit pattern without a code; needs 15 bits in the buffer
ABW_HD int decode(Bits& b, const uint16_t* count, const uint16_t* symbol, const uint16_t* fast, int fb)
{
	const uint32_t e = fast[b.buf & ((1u << fb) - 1)];
	if(e) {
		b.take((int)(e & 15));
		return (int)(e >> 4);
	}
	uint64_t bits = b.buf;
	int code = 0, first = 0, index = 0;
	for(int l = 1; l < 16; l++) {
		code |= (int)(bits & 1);
		bits >>= 1;
		const int c = count[l];
		if(code - c < first) {
			b.take(l);
			return symbol[index + (code - first)];
		}
		index += c;
		first += c;
		first <<= 1;
		code <<= 1;
	}
	return -1;
}

ABW_HD int codes(Bits& b, Tables& T, uint8_t* out, uint32_t cap, uint32_t& o)
{
	// base and extra bits of length and distance symbols (RFC 1951 3.2.5) computed rather than looked up: no tables in local memory
	for(;;) {
		if(b.pos > b.n + 8)
			return E_INPUT;
		b.refill();
		const int sym = decode(b, T.lcount, T.lsym, T.lfast, LFAST);
		if(sym < 0)
			return E_SYMBOL;
		if(sym < 256) {
			if(o >= cap)
				return E_OUTPUT;
			out[o++] = (uint8_t)sym;
		}
		else if(sym == 256)
			return OK;
		else {
			const int ls = sym - 257;
			if(ls >= 29)
				return E_SYMBOL;
			const int lx = (ls < 8 || ls == 28)? 0 : (ls - 4) >> 2;
			const uint32_t lb = (ls < 8)? 3u + ls : (ls == 28)? 258u : ((4u | (ls & 3)) << lx) + 3u;
			const uint32_t len = lb + b.take(lx);
			const int ds = decode(b, T.dcount, T.dsym, T.dfast, DFAST);
			if(ds < 0 || ds >= 30)
				return E_SYMBOL;
			if(b.cnt < 13)
				b.refill();
			const int dx = (ds < 4)? 0 : (ds >> 1) - 1;
			const uint32_t db = (ds < 4)? 1u + ds : ((2u | (ds & 1)) << dx) + 1u;
			const uint32_t dist = db + b.take(dx);
			if(dist > o)
				return E_DIST;
			if(len > cap - o)
				return E_OUTPUT;
			const uint8_t* src = out + (o - dist);
			for(uint32_t i = 0; i < len; i++)
				out[o + i] = src[i];
			o += len;
		}
	}
}

// Decodes the raw DEFLATE stream in[0 .. n) into out[0 .. cap); *out_len = bytes written.  Returns OK or an E_* code.
ABW_HD int inflate_raw(const uint8_t* in, uint32_t n, uint8_t* out, uint32_t cap, uint32_t* out_len, Tables& T)
{
	Bits b{in, n, 0, 0, 0};
	uint32_t o = 0;
	int last = 0, rc = OK;
	while(!last && rc == OK) {
		if(b.pos > b.n + 8) {
			rc = E_INPUT;
			break;
		}
		b.refill();
		last = (int)b.take(1);
		const uint32_t type = b.take(2);
		if(type == 0) {
			b.take(b.cnt & 7);
			const uint32_t len = b.take(16), nlen = b.take(16);
			if(len != (~nlen & 0xFFFFu)) {
				rc = E_STORED;
				break;
			}
			const uint32_t at = b.pos - (uint32_t)(b.cnt >> 3);      // the buffer holds whole bytes now
			if(at > n || len > n - at) {
				rc = E_INPUT;
				break;
			}
			if(len > cap - o) {
				rc = E_OUTPUT;
				break;
			}
			for(uint32_t i = 0; i < len; i++)
				out[o + i] = in[at + i];
			o += len;
			b.pos = at + len;
			b.buf = 0;
			b.cnt = 0;
		}
		else if(type == 1) {
			for(int s = 0; s < 288; s++)
				T.lens[s] = (s < 144)? 8 : (s < 256)? 9 : (s < 280)? 7 : 8;
			build(T.lens, 288, 1, T.lcount, T.lsym, T.lfast, LFAST);
			for(int s = 0; s < 32; s++)
				T.lens[s] = 5;
			build(T.lens, 32, 1, T.dcount, T.dsym, T.dfast, DFAST);
			rc = codes(b, T, out, cap, o);
		}
		else if(type == 2) {
			const int nlit = (int)b.take(5) + 257, ndist = (int)b.take(5) + 1, ncode = (int)b.take(4) + 4;
			if(nlit > 286 || ndist > 30) {
				rc = E_HEADER;
				break;
			}
			const char* order = "\x10\x11\x12\x00\x08\x07\x09\x06\x0a\x05\x0b\x04\x0c\x03\x0d\x02\x0e\x01\x0f";
			for(int i = 0; i < 19; i++)
				T.lens[i] = 0;
			for(int i = 0; i < ncode; i++) {
				if(b.cnt < 3)
					b.refill();
				T.lens[(uint8_t)order[i]] = (uint8_t)b.take(3);
			}
			// the code-length code lives in the distance tables until the distance code replaces it
			if((rc = build(T.lens, 19, 0, T.dcount, T.dsym, T.dfast, DFAST)) != OK)
				break;
			int idx = 0;
			while(idx < nlit + ndist) {
				if(b.pos > b.n + 8) {
					rc = E_INPUT;
					break;
				}
				b.refill();
				const int sym = decode(b, T.dcount, T.dsym, T.dfast, DFAST);
				if(sym < 0) {
					rc = E_SYMBOL;
					break;
				}
				if(sym < 16) {
					T.lens[idx++] = (uint8_t)sym;
					continue;
				}
				uint8_t v = 0;
				int rep;
				if(sym == 16) {
					if(idx == 0) {
						rc = E_HEADER;
						break;
					}
					v = T.lens[idx - 1];
					rep = 3 + (int)b.take(2);
				}
				else if(sym == 17)
					rep = 3 + (int)b.take(3);
				else
					rep = 11 + (int)b.take(7);
				if(idx + rep > nlit + ndist) {
					rc = E_HEADER;
					break;
				}
				while(rep--)
					T.lens[idx++] = v;
			}
			if(rc != OK)
				break;
			if(T.lens[256] == 0) {
				rc = E_HEADER;
				break;
			}
			if((rc = build(T.lens, nlit, 1, T.lcount, T.lsym, T.lfast, LFAST)) != OK)
				break;
			if((rc = build(T.lens + nlit, ndist, 1, T.dcount, T.dsym, T.dfast, DFAST)) != OK)
				break;
			rc = codes(b, T, out, cap, o);
		}
		else
			rc = E_BTYPE;
	}
	if(rc == OK && b.overrun())
		rc = E_INPUT;
	*out_len = o;
	return rc;
}

// ---- CRC-32 of gzip (reflected polynomial 0xEDB88320) ----
ABW_HD uint32_t crc32_table_entry(uint32_t i)
{
	uint32_t c = i;
	for(int k = 0; k < 8; k++)
		c = (c & 1)? (c >> 1) ^ 0xEDB88320u : c >> 1;
	return c;
}

// the CRC-32 of p[0 .. n) (table: the 256 entries of crc32_table_entry)
ABW_HD uint32_t crc32(const uint8_t* p, uint64_t n, const uint32_t* table)
{
	uint32_t c = 0xFFFFFFFFu;
	for(uint64_t i = 0; i < n; i++)
		c = table[(c ^ p[i]) & 0xFFu] ^ (c >> 8);
	return ~c;
}

// a * b modulo the polynomial (zlib's multmodp); a != 0
ABW_HD uint32_t crc32_multmodp(uint32_t a, uint32_t b)
{
	uint32_t m = 1u << 31, p = 0;
	for(;;) {
		if(a & m) {
			p ^= b;
			if((a & (m - 1)) == 0)
				break;
		}
		m >>= 1;
		b = (b & 1)? (b >> 1) ^ 0xEDB88320u : b >> 1;
	}
	return p;
}

// CRC-32 of A then B from crc(A), crc(B) and the length of B (zlib's crc32_combine)
ABW_HD uint32_t crc32_combine(uint32_t crc_a, uint32_t crc_b, uint64_t len_b)
{
	uint32_t op = 1u << 31, sq = 1u << 23;       // x^0, x^8
	for(; len_b; len_b >>= 1) {
		if(len_b & 1)
			op = crc32_multmodp(sq, op);
		sq = crc32_multmodp(sq, sq);
	}
	return crc32_multmodp(op, crc_a) ^ crc_b;
}

}  // namespace abw_inflate
