"""BAM input: the DEFLATE decoder of csrc/inflate.cuh against zlib (CPU, through a host build of the header), the synthetic BAM writer against a
test-local reader (CPU), and abw_bam_* against abw_parse_sam on the text `samtools view` prints for the same records (GPU)."""
import ctypes as C
import os
import struct
import subprocess
import zlib

import numpy as np
import pytest

from abawaca_b200 import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "abawaca_b200", "csrc")
BIN = os.path.join(ROOT, "abawaca_b200", "bin")

_DRIVER = r'''
#include "inflate.cuh"
extern "C" int drv_inflate(const uint8_t* in, uint32_t n, uint8_t* out, uint32_t cap, uint32_t* out_len)
{
	static abw_inflate::Tables T;
	return abw_inflate::inflate_raw(in, n, out, cap, out_len, T);
}
extern "C" uint32_t drv_crc32(const uint8_t* p, uint64_t n)
{
	uint32_t t[256];
	for(uint32_t i = 0; i < 256; i++)
		t[i] = abw_inflate::crc32_table_entry(i);
	return abw_inflate::crc32(p, n, t);
}
extern "C" uint32_t drv_crc32_combine(uint32_t a, uint32_t b, uint64_t len_b) { return abw_inflate::crc32_combine(a, b, len_b); }
'''


@pytest.fixture(scope="module")
def host_inflate(tmp_path_factory):
    d = tmp_path_factory.mktemp("inflate")
    src, lib = d / "drv.cpp", d / "drv.so"
    src.write_text(_DRIVER)
    subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-I", CSRC, str(src), "-o", str(lib)], check=True)
    L = C.CDLL(str(lib))
    L.drv_inflate.argtypes = [C.c_char_p, C.c_uint32, C.c_void_p, C.c_uint32, C.POINTER(C.c_uint32)]
    L.drv_crc32.argtypes = [C.c_char_p, C.c_uint64]
    L.drv_crc32.restype = C.c_uint32
    L.drv_crc32_combine.argtypes = [C.c_uint32, C.c_uint32, C.c_uint64]
    L.drv_crc32_combine.restype = C.c_uint32

    def inflate(data, cap):
        out = (C.c_uint8 * max(cap, 1))()
        n = C.c_uint32()
        rc = L.drv_inflate(bytes(data), len(data), out, cap, C.byref(n))
        return rc, bytes(out[:n.value])
    inflate.lib = L
    return inflate


def zlib_inflate(data):
    try:
        return zlib.decompress(bytes(data), -15)
    except zlib.error:
        return None


def _bam_payload():
    mg = synth.make_metagenome(30, 1, 2, 5)
    buf, _ = next(synth.sample_bam_records(mg, 0))
    return buf[:200000].tobytes()


def _payloads():
    rng = np.random.default_rng(3)
    rnd = rng.integers(0, 256, 70000, dtype=np.uint8).tobytes()
    far = rng.integers(0, 256, 32768, dtype=np.uint8).tobytes()
    return {
        "random": rnd,
        "run": b"a" * 70000,                                       # distance 1, overlapping, length 258
        "period3": b"xyz" * 20000,
        "far": far + far + far[:1000],                            # distance 32768
        "bam": _bam_payload(),
        "text": b"".join(b"r%d\t%d\t*\t0\n" % (i, i * 7) for i in range(4000)),
        "empty": b"",
    }


PAYLOADS = _payloads()
SETTINGS = [(0, zlib.Z_DEFAULT_STRATEGY), (1, zlib.Z_DEFAULT_STRATEGY), (6, zlib.Z_DEFAULT_STRATEGY), (9, zlib.Z_DEFAULT_STRATEGY),
            (6, zlib.Z_FILTERED), (6, zlib.Z_HUFFMAN_ONLY), (6, zlib.Z_RLE), (6, zlib.Z_FIXED)]


def _deflate(data, level, strategy, flushes=()):
    c = zlib.compressobj(level, zlib.DEFLATED, -15, 9, strategy)
    out, o = [], 0
    for at, mode in flushes:
        out += [c.compress(data[o:at]), c.flush(mode)]
        o = at
    return b"".join(out + [c.compress(data[o:]), c.flush()])


@pytest.mark.parametrize("name", sorted(PAYLOADS))
@pytest.mark.parametrize("level,strategy", SETTINGS)
def test_host_inflate_matches_zlib(host_inflate, name, level, strategy):
    data = PAYLOADS[name]
    comp = _deflate(data, level, strategy)
    assert zlib_inflate(comp) == data
    rc, out = host_inflate(comp, len(data))
    assert rc == 0 and out == data
    if data:
        assert host_inflate(comp, len(data) - 1)[0] != 0            # output past the cap (a block's ISIZE)


@pytest.mark.parametrize("level", [0, 6])
def test_host_inflate_flushes(host_inflate, level):
    data = PAYLOADS["bam"][:60000]
    comp = _deflate(data, level, zlib.Z_DEFAULT_STRATEGY, [(100, zlib.Z_SYNC_FLUSH), (100, zlib.Z_FULL_FLUSH), (30000, zlib.Z_SYNC_FLUSH),
                                                           (50000, zlib.Z_FULL_FLUSH)])
    assert zlib_inflate(comp) == data
    assert host_inflate(comp, len(data)) == (0, data)


def test_host_crc32(host_inflate):
    L = host_inflate.lib
    for data in (b"", b"a", PAYLOADS["random"], PAYLOADS["bam"][:65536]):
        assert L.drv_crc32(data, len(data)) == zlib.crc32(data)
    a, b = PAYLOADS["random"][:12345], PAYLOADS["bam"][:54321]
    assert L.drv_crc32_combine(zlib.crc32(a), zlib.crc32(b), len(b)) == zlib.crc32(a + b)
    assert L.drv_crc32_combine(zlib.crc32(a), 0, 0) == zlib.crc32(a)


# ---- hand-built streams -----------------------------------------------------------------------------------------------------
class BitWriter:
    def __init__(self):
        self.v, self.n = 0, 0

    def bits(self, value, n):
        self.v |= (value & ((1 << n) - 1)) << self.n
        self.n += n
        return self

    def code(self, code, length):              # Huffman codes go in from their most significant bit
        for i in range(length - 1, -1, -1):
            self.bits((code >> i) & 1, 1)
        return self

    def align(self):
        self.n += (-self.n) % 8
        return self

    def bytes(self):
        return self.v.to_bytes((self.n + 7) // 8, "little")


def canon(lengths):
    """canonical codes {symbol: (code, length)}"""
    bl = [0] * 16
    for ln in lengths:
        bl[ln] += 1
    bl[0] = 0
    nxt, code = [0] * 16, 0
    for b in range(1, 16):
        code = (code + bl[b - 1]) << 1
        nxt[b] = code
    out = {}
    for s, ln in enumerate(lengths):
        if ln:
            out[s] = (nxt[ln], ln)
            nxt[ln] += 1
    return out


CL_ORDER = [16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15]
CL_LENS = [4] * 13 + [5] * 6                   # a complete code-length code over the 19 symbols


def dyn_block(w, lit, dist, cl=CL_LENS, final=1, nlit=None, ndist=None, lens_syms=None):
    """header of a dynamic block: lit/dist code lengths written one symbol each (or the given code-length symbols); returns the two codes"""
    nl = len(lit) if nlit is None else nlit
    nd = len(dist) if ndist is None else ndist
    w.bits(final, 1).bits(2, 2).bits(nl - 257, 5).bits(nd - 1, 5).bits(19 - 4, 4)
    for s in CL_ORDER:
        w.bits(cl[s], 3)
    cc = canon(cl)
    for item in (lens_syms if lens_syms is not None else [(x,) for x in list(lit) + list(dist)]):
        w.code(*cc[item[0]])
        if len(item) > 1:
            w.bits(item[1], item[2])
    return canon(list(lit)), canon(list(dist))


def fixed(w, final=1):
    w.bits(final, 1).bits(1, 2)
    return canon([8] * 144 + [9] * 112 + [7] * 24 + [8] * 8), canon([5] * 32)


def _lit_lens(extra=None):
    lens = [0] * 257
    for s in b"abc":
        lens[s] = 2
    lens[256] = 2
    if extra:
        lens += extra
    return lens


def _stream_cases():
    cases = {}
    w = BitWriter().bits(1, 1).bits(3, 2)
    cases["btype3"] = w.bytes() + b"\0\0"
    cases["stored_ok"] = BitWriter().bits(1, 1).bits(0, 2).align().bits(3, 16).bits(0xFFFC, 16).bytes() + b"xyz"
    cases["stored_bad_nlen"] = BitWriter().bits(1, 1).bits(0, 2).align().bits(3, 16).bits(0xFFFD, 16).bytes() + b"xyz"
    cases["stored_short"] = BitWriter().bits(1, 1).bits(0, 2).align().bits(3, 16).bits(0xFFFC, 16).bytes() + b"xy"
    cases["empty_stored_then_fixed"] = BitWriter().bits(0, 1).bits(0, 2).align().bits(0, 16).bits(0xFFFF, 16).bits(1, 1).bits(1, 2).bits(0, 7).bytes()

    def dyn(name, lit, dist, body, **kw):
        w = BitWriter()
        lc, dc = dyn_block(w, lit, dist, **kw)
        body(w, lc, dc)
        cases[name] = w.bytes()

    def abc_eob(w, lc, dc):
        for s in b"abca":
            w.code(*lc[s])
        w.code(*lc[256])

    dyn("dyn_ok", _lit_lens(), [1, 1], abc_eob)
    dyn("dyn_cl_oversubscribed", _lit_lens(), [1, 1], abc_eob, cl=[3] * 19)
    dyn("dyn_cl_incomplete", _lit_lens(), [1, 1], abc_eob, cl=[4] * 13 + [5] * 5 + [0])
    over = _lit_lens()
    over[ord("d")] = 2
    over[ord("e")] = 2
    dyn("dyn_lit_oversubscribed", over, [1, 1], abc_eob)
    inc = _lit_lens()
    inc[ord("c")] = 3
    dyn("dyn_lit_incomplete", inc, [1, 1], abc_eob)
    only_eob = [0] * 256 + [1]
    dyn("dyn_single_eob_code", only_eob, [1, 1], lambda w, lc, dc: w.code(*lc[256]))
    no_eob = _lit_lens()
    no_eob[256] = 0
    no_eob[ord("d")] = 2
    dyn("dyn_missing_eob", no_eob, [1, 1], lambda w, lc, dc: [w.code(*lc[s]) for s in b"abd"])
    # matches: literal 'a', 'b', then length 3 (symbol 257) at distance 2 (dist symbol 1), twice; distance codes vary
    lit_m = _lit_lens([2])                      # symbol 257 too: 5 codes of length 2 would over-subscribe, so 'c' goes
    lit_m[ord("c")] = 0

    def match(dsym, dist_extra=None):
        def body(w, lc, dc):
            w.code(*lc[ord("a")]).code(*lc[ord("b")])
            for _ in range(2):
                w.code(*lc[257]).code(*dc[dsym])
                if dist_extra:
                    w.bits(*dist_extra)
            w.code(*lc[256])
        return body

    dyn("dyn_match_ok", lit_m, [1, 1], match(1))
    dyn("dyn_single_distance_code", lit_m, [0, 1], match(1))
    dyn("dyn_single_distance_code_unused_pattern", lit_m, [0, 1], lambda w, lc, dc: (w.code(*lc[ord("a")]), w.code(*lc[257]), w.bits(1, 1), w.code(*lc[256])))
    dyn("dyn_empty_distance_code", _lit_lens(), [0], abc_eob)
    dyn("dyn_distance_too_far", lit_m, [0, 0, 1, 1], match(2))              # distance 3 after two bytes
    dyn("dyn_dist_oversubscribed", lit_m, [1, 1, 1], match(1))
    dyn("dyn_dist_incomplete", lit_m, [2, 2, 2], match(1))
    dyn("dyn_hlit_287", _lit_lens() + [0] * 30, [1, 1], abc_eob)
    dyn("dyn_hlit_288", _lit_lens() + [0] * 31, [1, 1], abc_eob)
    dyn("dyn_hdist_31", _lit_lens(), [1, 1] + [0] * 29, abc_eob)
    dyn("dyn_hdist_32", _lit_lens(), [1, 1] + [0] * 30, abc_eob)
    dyn("dyn_hdist_30", _lit_lens(), [1, 1] + [0] * 28, abc_eob)
    # repeat codes: 16 first (nothing to repeat), 18 past the end, and a valid mix
    lens = _lit_lens()
    seq, i = [], 0
    full = lens + [1, 1]
    while i < len(full):
        j = i
        while j < len(full) and full[j] == full[i]:
            j += 1
        run = j - i
        if full[i] == 0 and run >= 11:
            k = min(run, 138)
            seq.append((18, k - 11, 7))
            i += k
        elif full[i] == 0 and run >= 3:
            k = min(run, 10)
            seq.append((17, k - 3, 3))
            i += k
        elif run >= 4:
            seq.append((full[i],))
            k = min(run - 1, 6)
            seq.append((16, k - 3, 2))
            i += 1 + k
        else:
            seq.append((full[i],))
            i += 1
    dyn("dyn_repeats_ok", lens, [1, 1], abc_eob, lens_syms=seq)
    dyn("dyn_repeat16_first", lens, [1, 1], abc_eob, lens_syms=[(16, 0, 2)] + seq)
    dyn("dyn_repeat18_past_end", lens, [1, 1], abc_eob, lens_syms=seq[:-1] + [(18, 0, 7)])
    # fixed code: literal/length 286 and 287, distance 30 and 31, a distance before the start, a valid run
    for s in (286, 287):
        w = BitWriter()
        lc, dc = fixed(w)
        w.code(*lc[ord("a")]).code(*lc[s]).code(*dc[0]).code(*lc[256])
        cases[f"fixed_sym{s}"] = w.bytes()
    for d in (30, 31):
        w = BitWriter()
        lc, dc = fixed(w)
        w.code(*lc[ord("a")]).code(*lc[257]).code(*dc[d]).bits(0, 13).code(*lc[256])
        cases[f"fixed_dist{d}"] = w.bytes()
    w = BitWriter()
    lc, dc = fixed(w)
    w.code(*lc[ord("a")]).code(*lc[285]).code(*dc[0]).code(*lc[257]).code(*dc[1]).code(*lc[256])
    cases["fixed_long_match"] = w.bytes()
    w = BitWriter()
    lc, dc = fixed(w)
    w.code(*lc[ord("a")]).code(*lc[257]).code(*dc[1]).code(*lc[256])        # distance 2 after one byte
    cases["fixed_too_far"] = w.bytes()
    w = BitWriter()
    lc, dc = fixed(w)
    w.code(*lc[ord("a")]).code(*lc[284]).bits(31, 5).code(*dc[0]).code(*lc[256])     # 227 + 31 = 258 through symbol 284, as zlib accepts
    cases["fixed_284_258"] = w.bytes()
    return cases


STREAMS = _stream_cases()


@pytest.mark.parametrize("name", sorted(STREAMS))
def test_host_inflate_rejects_what_zlib_rejects(host_inflate, name):
    data = STREAMS[name]
    ref = zlib_inflate(data)
    rc, out = host_inflate(data, 1 << 16)
    assert (rc == 0) == (ref is not None), (rc, ref)
    if ref is not None:
        assert out == ref


def test_hand_built_streams_cover_both_outcomes():
    ok = [k for k, v in STREAMS.items() if zlib_inflate(v) is not None]
    assert {"stored_ok", "dyn_ok", "dyn_match_ok", "dyn_single_eob_code", "dyn_single_distance_code", "dyn_empty_distance_code", "dyn_repeats_ok",
            "dyn_hdist_30", "fixed_284_258", "fixed_long_match", "empty_stored_then_fixed"} <= set(ok)
    assert {"btype3", "stored_bad_nlen", "dyn_cl_oversubscribed", "dyn_cl_incomplete", "dyn_lit_oversubscribed", "dyn_lit_incomplete", "dyn_missing_eob",
            "dyn_distance_too_far", "dyn_hlit_287", "dyn_hlit_288", "dyn_hdist_31", "fixed_sym286", "fixed_sym287", "fixed_dist30", "fixed_dist31",
            "fixed_too_far", "dyn_repeat16_first", "dyn_repeat18_past_end", "dyn_single_distance_code_unused_pattern"}.isdisjoint(ok)


@pytest.mark.parametrize("name", ["dyn_repeats_ok", "dyn_match_ok", "stored_ok", "fixed_284_258"])
def test_host_inflate_truncated(host_inflate, name):
    data = STREAMS[name]
    for k in range(len(data)):
        assert zlib_inflate(data[:k]) is None
        assert host_inflate(data[:k], 1 << 16)[0] != 0, k


# ---- a test-local BAM reader and `samtools view` formatter ------------------------------------------------------------------
def read_bgzf(data):
    """(decoded stream, per-block ISIZE) of a BGZF file"""
    out, sizes, o = [], [], 0
    while o < len(data):
        assert data[o:o + 4] == b"\x1f\x8b\x08\x04" and data[o + 12:o + 16] == b"BC\x02\x00"
        bsize = struct.unpack_from("<H", data, o + 16)[0] + 1
        crc, isize = struct.unpack_from("<II", data, o + bsize - 8)
        dec = zlib.decompress(data[o + 18:o + bsize - 8], -15)
        assert len(dec) == isize and zlib.crc32(dec) == crc
        out.append(dec)
        sizes.append(isize)
        o += bsize
    return b"".join(out), sizes


def parse_bam(data):
    """(reference names, records as dicts) of a BAM file"""
    s, _ = read_bgzf(data)
    assert s[:4] == b"BAM\1"
    lt = struct.unpack_from("<i", s, 4)[0]
    o = 8 + lt
    nref = struct.unpack_from("<i", s, o)[0]
    o += 4
    refs = []
    for _ in range(nref):
        ln = struct.unpack_from("<i", s, o)[0]
        refs.append(s[o + 4:o + 4 + ln].split(b"\0")[0].decode())
        o += 8 + ln
    recs = []
    while o < len(s):
        bs = struct.unpack_from("<i", s, o)[0]
        r = s[o + 4:o + 4 + bs]
        refID, pos, lrn, mapq, _, ncig, flag, lseq, mref, mpos, tlen = struct.unpack_from("<iiBBHHHiiii", r, 0)
        p = 32
        name = r[p:p + lrn - 1].decode()
        p += lrn
        cigar = [(v & 15, v >> 4) for v in struct.unpack_from(f"<{ncig}I", r, p)]
        p += 4 * ncig
        packed = r[p:p + (lseq + 1) // 2]
        seq = "".join("=ACMGRSVTWYHKDBN"[(packed[i // 2] >> (4 * (1 - i % 2))) & 15] for i in range(lseq))
        p += (lseq + 1) // 2
        qual = r[p:p + lseq]
        p += lseq
        aux = []
        while p < len(r):
            tag, t = r[p:p + 2].decode(), chr(r[p + 2])
            p += 3
            if t in "AcC":
                v = chr(r[p]) if t == "A" else struct.unpack_from("<" + t.replace("C", "B").replace("c", "b"), r, p)[0]
                p += 1
            elif t in "sS":
                v = struct.unpack_from("<" + ("h" if t == "s" else "H"), r, p)[0]
                p += 2
            elif t in "iIf":
                v = struct.unpack_from("<" + t, r, p)[0]
                p += 4
            elif t in "ZH":
                e = r.index(b"\0", p)
                v = r[p:e].decode()
                p = e + 1
            elif t == "B":
                sub, cnt = chr(r[p]), struct.unpack_from("<I", r, p + 1)[0]
                sz = {"c": 1, "C": 1, "s": 2, "S": 2, "i": 4, "I": 4, "f": 4}[sub]
                v = (sub, list(struct.unpack_from(f"<{cnt}{ {'c': 'b', 'C': 'B'}.get(sub, sub) if sub not in 'sS' else ('h' if sub == 's' else 'H')}", r, p + 5)))
                p += 5 + cnt * sz
            else:
                raise AssertionError(t)
            aux.append((tag, t, v))
        assert p == len(r)
        recs.append(dict(refID=refID, pos=pos, name=name, mapq=mapq, flag=flag, cigar=cigar, seq=seq, qual=qual, aux=aux, mref=mref, mpos=mpos, tlen=tlen))
        o += 4 + bs
    assert o == len(s)
    return refs, recs


def sam_text(refs, recs):
    """the lines `samtools view` prints, for the fields abw_parse_sam reads (a CG:B:I tag under the long-CIGAR convention replaces the CIGAR)"""
    lines = []
    for r in recs:
        cigar, aux = r["cigar"], r["aux"]
        cg = next((a for a in aux if a[0] == "CG"), None)
        if (cigar and r["refID"] >= 0 and r["pos"] >= 0 and cigar[0] == (4, len(r["seq"])) and cg and cg[1] == "B" and cg[2][0] in "Ii"):
            cigar = [(v & 15, v >> 4) for v in cg[2][1]]
            aux = [a for a in aux if a is not cg]
        ctext = "".join(f"{ln}{'MIDNSHP=XBB?????'[op]}" for op, ln in cigar) or "*"
        fields = []
        for tag, t, v in aux:
            if t == "B":
                fields.append(f"{tag}:B:{v[0]}" + "".join(f",{x:g}" if v[0] == "f" else f",{x}" for x in v[1]))
            elif t in "cCsSiI":
                fields.append(f"{tag}:i:{v}")
            elif t == "f":
                fields.append(f"{tag}:f:{v:g}")
            else:
                fields.append(f"{tag}:{t}:{v}")
        rname = refs[r["refID"]] if r["refID"] >= 0 else "*"
        qual = "*" if not r["qual"] or r["qual"][0] == 0xFF else "".join(chr(q + 33) for q in r["qual"])
        lines.append("\t".join([r["name"], str(r["flag"]), rname, str(r["pos"] + 1), str(r["mapq"]), ctext, "*", str(r["mpos"] + 1), str(r["tlen"]),
                                r["seq"] or "*", qual] + fields))
    return ("\n".join(lines) + "\n").encode() if lines else b""


def test_synth_bam_round_trip(tmp_path):
    mg = synth.make_metagenome(40, 2, 3, 17, bad_read_frac=0.1)
    for aligned, cut in ((True, None), (False, None), (False, 777)):
        path = str(tmp_path / f"rt_{aligned}_{cut}.bam")
        synth.write_bam(path, mg, 1, aligned=aligned, cut=cut, level=1)
        data = open(path, "rb").read()
        _, sizes = read_bgzf(data)
        assert sizes[-1] == 0 and max(sizes) <= 0xff00
        refs, recs = parse_bam(data)
        assert refs == mg.names
        rec = mg.reads[1]
        assert len(recs) == rec.size
        flag = rec["flag_nsnps"] & 0xFFFF
        unm = (flag & 4) != 0
        assert [r["flag"] for r in recs] == flag.tolist()
        assert [r["refID"] for r in recs] == np.where(unm, -1, rec["scaf"].astype(np.int64)).tolist()
        assert [r["pos"] for r in recs] == np.where(unm, -1, rec["pos0"].astype(np.int64)).tolist()
        assert all(len(r["seq"]) == n for r, n in zip(recs, rec["len"].tolist()))
        k = int(np.flatnonzero(~unm)[0])
        s0 = mg.scaffold(int(rec["scaf"][k]))[int(rec["pos0"][k]):int(rec["pos0"][k]) + int(rec["len"][k])].tobytes().decode()
        assert recs[k]["seq"] == s0 and recs[k]["cigar"] == [(0, int(rec["len"][k]))]
        nsn = (rec["flag_nsnps"] >> 16).tolist()
        for r, u, ns, ln in zip(recs, unm.tolist(), nsn, rec["len"].tolist()):
            assert r["aux"] == ([] if u else [("MD", "Z", synth._md_text(ln, ns))])
        if aligned:
            # htslib's layout: every block after the header's starts at a record
            s, sizes = read_bgzf(data)
            starts, o = set(), struct.unpack_from("<i", s, 4)[0] + 12
            for n in refs:
                o += 8 + len(n) + 1
            hdr = o
            while o < len(s):
                starts.add(o)
                o += 4 + struct.unpack_from("<i", s, o)[0]
            assert sizes[0] == hdr
            assert all(b in starts for b in np.cumsum(sizes)[:-2].tolist()[1:])


# ---- GPU: abw_bam_* against abw_parse_sam ------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def ctx():
    from abawaca_b200 import capi
    c = capi.Context(0)
    yield c
    c.close()


def bgzf_file(stream_parts, level=6, sizes=None, eof=True):
    """BGZF blocks of the given payloads (bytes each), plus the EOF block"""
    return b"".join(synth._bgzf_block(p, level, zlib.Z_DEFAULT_STRATEGY) for p in stream_parts) + (synth.BGZF_EOF if eof else b"")


def cut_stream(stream, sizes):
    out, o, i = [], 0, 0
    while o < len(stream):
        k = sizes[i % len(sizes)]
        out.append(stream[o:o + k])
        o += k
        i += 1
    return out


def feed_all(ctx, names, data, split=None, rng=None):
    from abawaca_b200 import pipeline
    r = pipeline.BamReader(ctx, names)
    try:
        if split == "random":
            cuts = np.sort(rng.integers(0, len(data) + 1, 40))
            pieces = [data[a:b] for a, b in zip([0] + cuts.tolist(), cuts.tolist() + [len(data)])]
        else:
            k = split or len(data) or 1
            pieces = [data[o:o + k] for o in range(0, len(data), k)]
        for p in pieces:
            r.feed(p)
        return r.to_host()
    finally:
        r.close()


def sam_records(ctx, names, data):
    from abawaca_b200 import pipeline
    refs, recs = parse_bam(data)
    p = pipeline.SamParser(ctx, names)
    try:
        return p.parse_to_host(sam_text(refs, recs))
    finally:
        p.close()


def check_bam(ctx, names, data, splits=(None,), rng=None):
    want = sam_records(ctx, names, data)
    for split in splits:
        got = feed_all(ctx, names, data, split, rng)
        assert got.size == want.size, split
        assert np.array_equal(got, want), split
    return want


def _aux(tag, t, v):
    if t == "A":
        return tag.encode() + b"A" + v.encode()
    if t in "cCsSiIf":
        return tag.encode() + t.encode() + struct.pack("<" + {"c": "b", "C": "B", "s": "h", "S": "H", "i": "i", "I": "I", "f": "f"}[t], v)
    if t in "ZH":
        return tag.encode() + t.encode() + v.encode() + b"\0"
    sub, vals = v
    return tag.encode() + b"B" + sub.encode() + struct.pack("<I", len(vals)) + struct.pack("<" + str(len(vals)) + {"c": "b", "C": "B", "s": "h", "S": "H"}.get(sub, sub), *vals)


EDGE_REFS = ["chrA", "chrB", "not_in_assembly", "chrC"]
EDGE_LENS = [100000, 5000, 3000, 80000]


def edge_records():
    S = "ACGTTGCAAC" * 15
    md = lambda s: _aux("MD", "Z", s)            # noqa: E731
    R = synth.bam_record
    recs = [
        R(0, 99, "plain", 0, [(0, 150)], S, list(range(150)), md("150")),
        R(0, 5, "no_seq", 0, [(0, 150)], "", None, md("150")),                     # l_seq 0: SEQ "*", length 1
        R(-1, -1, "unmapped", 4, [], S[:50]),
        R(-1, 17, "unmapped_pos", 4, [], S[:50], None, md("50")),
        R(2, 10, "unknown_name", 0, [(0, 50)], S[:50], None, md("50")),
        R(1, 0, "md_in_value", 0, [(0, 50)], S[:50], None, _aux("XA", "Z", "foo MD:Z:3A2^GG44 bar")),
        R(1, 1, "md_space", 0, [(0, 50)], S[:50], None, md("10A10 C4")),
        R(1, 2, "md_not_z", 0, [(0, 50)], S[:50], None, _aux("MD", "i", 5) + _aux("XB", "Z", "x") + md("2T47")),
        R(1, 3, "md_after_all_types", 0, [(0, 20), (1, 5), (0, 25)], S[:50], None,
          _aux("XA", "A", "q") + _aux("Xc", "c", -5) + _aux("XC", "C", 200) + _aux("Xs", "s", -300) + _aux("XS", "S", 60000) + _aux("Xi", "i", -70000) +
          _aux("XI", "I", 4000000000) + _aux("Xf", "f", 1.5) + _aux("XH", "H", "1AE301") + _aux("Bc", "B", ("c", [-1, 2])) + _aux("BC", "B", ("C", [255])) +
          _aux("Bs", "B", ("s", [-2, 3, 4])) + _aux("BS", "B", ("S", [])) + _aux("Bi", "B", ("i", [-7])) + _aux("BI", "B", ("I", [7, 8])) +
          _aux("Bf", "B", ("f", [0.5, 2.0])) + md("5A19^T25")),
        R(3, 7, "ins_no_md", 0, [(0, 10), (1, 3), (0, 37)], S[:50]),
        R(3, 8, "sixteen", 0, [(0, 50)], S[:50], None, md("0" + "A0" * 15 + "A34")),
        R(3, 9, "huge_deletion", 0, [(0, 25), (2, 70000), (0, 25)], S[:50], None, md("25^" + "ACGT" * 17500 + "25")),
        # the long-CIGAR convention: a soft clip of the whole read, the real CIGAR in CG:B:I
        R(0, 300, "cg", 0, [(4, 50), (3, 100)], S[:50], None, md("45") + _aux("CG", "B", ("I", [(20 << 4) | 0, (2 << 4) | 1, (3 << 4) | 1, (25 << 4) | 0]))),
        R(0, 301, "cg_i", 0, [(4, 50)], S[:50], None, _aux("CG", "B", ("i", [(48 << 4) | 0, (2 << 4) | 1])) + md("48")),
        R(0, 302, "cg_wrong_clip", 0, [(4, 49), (0, 1)], S[:50], None, _aux("CG", "B", ("I", [(2 << 4) | 1])) + md("50")),
        R(-1, 303, "cg_no_ref", 0, [(4, 50)], S[:50], None, _aux("CG", "B", ("I", [(2 << 4) | 1])) + md("50")),
        R(0, 304, "cg_not_first", 0, [(4, 50)], S[:50], None, _aux("CG", "Z", "x") + _aux("CG", "B", ("I", [(2 << 4) | 1])) + md("50")),
        R(0, 305, "cg_short_type", 0, [(4, 50)], S[:50], None, _aux("CG", "B", ("S", [(2 << 4) | 1])) + md("50")),
        R(1, 4, "flag_high", 0xFFFF & 0x900, [(0, 50)], S[:50], None, md("50")),
    ]
    return recs


def edge_bam(level=6):
    stream = synth.bam_header(EDGE_REFS, EDGE_LENS) + b"".join(edge_records())
    return stream, bgzf_file(cut_stream(stream, [0xff00]), level)


@pytest.mark.gpu
@pytest.mark.parametrize("names", [["chrA", "chrB", "chrC"], ["*", "chrA", "chrB", "chrC"]])
def test_edge_records(ctx, names):
    _, data = edge_bam()
    want = check_bam(ctx, names, data, splits=(None, 1, 17, 65537))
    by = {r["name"]: i for i, r in enumerate(parse_bam(data)[1])}
    nsn = want["flag_nsnps"] >> 16
    assert want["len"][by["no_seq"]] == 1
    assert nsn[by["md_in_value"]] == 3 and nsn[by["md_space"]] == 1 and nsn[by["md_not_z"]] == 1 and nsn[by["md_after_all_types"]] == 2 + 1
    assert nsn[by["sixteen"]] == 16 and nsn[by["huge_deletion"]] == 0xFFFF and nsn[by["ins_no_md"]] == 0
    assert nsn[by["cg"]] == 2 and nsn[by["cg_i"]] == 1 and nsn[by["cg_wrong_clip"]] == 0 and nsn[by["cg_no_ref"]] == 0 and nsn[by["cg_not_first"]] == 0
    assert want["scaf"][by["unknown_name"]] == 0xFFFFFFFF and want["pos0"][by["unmapped"]] == 0xFFFFFFFF
    assert want["scaf"][by["unmapped"]] == (0 if names[0] == "*" else 0xFFFFFFFF)


def _sample_stream(nscaf=60, seed=9, bad=0.05):
    mg = synth.make_metagenome(nscaf, 1, 3, seed, bad_read_frac=bad)
    buf, size = next(synth.sample_bam_records(mg, 0))
    return mg, synth.bam_header(mg.names, np.diff(mg.offsets.astype(np.int64))), buf.tobytes(), size


@pytest.mark.gpu
@pytest.mark.parametrize("cut", [[1], [3], [7], [4093], [2, 5, 11, 64, 301, 0xff00]])
def test_records_cross_blocks(ctx, cut):
    mg, hdr, recs, size = _sample_stream(nscaf=8 if cut[0] < 4 else 40)
    stream = hdr + recs
    if cut[0] < 4:
        stream = hdr + recs[:int(np.cumsum(size)[400])]
    parts = cut_stream(stream, cut)
    data = bgzf_file(parts, level=1)
    starts = len(hdr) + np.concatenate([[0], np.cumsum(size)])
    bounds = np.cumsum([len(p) for p in parts])
    inside = bounds[(bounds > starts[0]) & (bounds < len(stream))]
    k = np.searchsorted(starts, inside, side="right") - 1
    if max(cut) < 8:
        assert set(range(int(np.diff(starts).min()))) <= set((inside - starts[k]).tolist())   # blocks end at every offset of a record
    if cut[0] < len(hdr):
        assert any(b < len(hdr) for b in bounds)                         # and inside the header
    check_bam(ctx, mg.names, data, splits=(None, "random") if cut[0] < 8 else (None, 17, "random"), rng=np.random.default_rng(len(cut)))


@pytest.mark.gpu
def test_empty_blocks_and_eof_blocks(ctx):
    mg, hdr, recs, _ = _sample_stream()
    parts = cut_stream(hdr + recs, [1000, 0xff00, 5])
    parts = [x for p in parts for x in (p, b"", b"")] + [b""]
    data = bgzf_file(parts) + synth.BGZF_EOF
    check_bam(ctx, mg.names, data, splits=(None, 1 << 16, "random"), rng=np.random.default_rng(2))


@pytest.mark.gpu
@pytest.mark.parametrize("aligned,level,strategy", [(True, 6, zlib.Z_DEFAULT_STRATEGY), (False, 1, zlib.Z_DEFAULT_STRATEGY), (True, 9, zlib.Z_FILTERED),
                                                    (False, 6, zlib.Z_RLE)])
def test_larger_sample(ctx, tmp_path, aligned, level, strategy):
    """a sample of over 64 MB decoded (several batches), against its SAM text and the generator"""
    mg = synth.make_metagenome(1500, 1, 6, 77)
    path = str(tmp_path / "s.bam")
    synth.write_bam(path, mg, 0, aligned=aligned, level=level, strategy=strategy)
    data = open(path, "rb").read()
    s, sizes = read_bgzf(data)
    assert len(s) > 64 << 20
    got = feed_all(ctx, mg.names, data, 64 << 20)
    ref = mg.reads[0]
    unm = (ref["flag_nsnps"] & 4) != 0
    want = ref.copy()
    want["scaf"][unm] = 0xFFFFFFFF
    want["pos0"][unm] = 0xFFFFFFFF
    assert np.array_equal(got, want)
    if level == 6 and aligned:
        from abawaca_b200 import pipeline
        p = pipeline.SamParser(ctx, mg.names)
        sam = synth.write_reference_inputs(mg, str(tmp_path))["sams"][0]
        assert np.array_equal(got, p.parse_to_host(open(sam, "rb").read()))
        p.close()


MALFORMED = {}


def _malformed():
    mg, hdr, recs, size = _sample_stream(nscaf=20)
    stream = hdr + recs
    good = bgzf_file(cut_stream(stream, [3000]))
    blk1 = struct.unpack_from("<H", good, 16)[0] + 1          # the first block's size
    out = {}

    def patch(data, at, b):
        return data[:at] + bytes(b) + data[at + len(b):]
    out["id1"] = patch(good, blk1, [30])
    out["cm"] = patch(good, blk1 + 2, [7])
    out["flg"] = patch(good, blk1 + 3, [0])
    out["xlen"] = patch(good, blk1 + 10, [7])
    out["si"] = patch(good, blk1 + 12, [ord("X")])
    out["slen"] = patch(good, blk1 + 14, [3])
    out["bsize_past_end"] = good[:blk1 + 100]
    out["bsize_tiny"] = patch(good, blk1 + 16, [10, 0])
    out["isize_big"] = patch(good, blk1 - 4, list(struct.pack("<I", 70000)))
    out["isize_short"] = patch(good, blk1 - 4, list(struct.pack("<I", 2999)))
    out["isize_long"] = patch(good, blk1 - 4, list(struct.pack("<I", 3001)))
    out["crc"] = patch(good, blk1 - 8, [good[blk1 - 8] ^ 1])
    for name in ("btype3", "stored_bad_nlen", "dyn_cl_incomplete", "dyn_lit_oversubscribed", "fixed_sym286", "fixed_dist30", "dyn_distance_too_far",
                 "dyn_single_distance_code_unused_pattern"):
        cdata = STREAMS[name]
        out["deflate_" + name] = good[:blk1] + struct.pack("<BBBBIBBHBBHH", 31, 139, 8, 4, 0, 0, 255, 6, 66, 67, 2, len(cdata) + 25) + cdata + \
            struct.pack("<II", 0, 0) + good[blk1:]
    out["magic"] = bgzf_file(cut_stream(b"BAM\2" + stream[4:], [0xff00]))
    out["l_text"] = bgzf_file(cut_stream(stream[:4] + struct.pack("<i", -1) + stream[8:], [0xff00]))
    at = 8 + struct.unpack_from("<i", stream, 4)[0]
    out["n_ref"] = bgzf_file(cut_stream(stream[:at] + struct.pack("<i", -20) + stream[at + 4:], [0xff00]))
    o = len(hdr)
    bs = struct.unpack_from("<i", stream, o)[0]
    out["block_size"] = bgzf_file(cut_stream(stream[:o] + struct.pack("<i", bs - 1) + stream[o + 4:], [0xff00]))
    out["l_seq"] = bgzf_file(cut_stream(stream[:o + 20] + struct.pack("<i", 100000) + stream[o + 24:], [0xff00]))
    out["refid"] = bgzf_file(cut_stream(stream[:o + 4] + struct.pack("<i", 20) + stream[o + 8:], [0xff00]))
    rec0 = stream[o:o + 4 + bs]
    junk = struct.pack("<i", bs + 2) + rec0[4:] + b"X\0"
    out["aux_junk"] = bgzf_file(cut_stream(stream[:o] + junk + stream[o + 4 + bs:], [0xff00]))
    bad_md = synth.bam_record(0, 1, "bad_md", 0, [(0, 10)], "ACGTACGTAC", None, _aux("MD", "Z", "5a4"))
    out["md"] = bgzf_file(cut_stream(stream + bad_md, [0xff00]))
    out["ends_in_record"] = bgzf_file(cut_stream(stream[:-10], [0xff00]))
    out["ends_in_header"] = bgzf_file(cut_stream(hdr[:len(hdr) - 3], [0xff00]))
    out["empty_file"] = b""
    return good, stream, out


@pytest.mark.gpu
def test_malformed_files(ctx):
    from abawaca_b200 import capi
    good, stream, bad = _malformed()
    mg, _, _, _ = _sample_stream(nscaf=20)
    feed_all(ctx, mg.names, good)
    for name, data in bad.items():
        with pytest.raises(capi.AbwError) as e:
            feed_all(ctx, mg.names, data)
        assert "status 2" in str(e.value), name
        if name == "md":
            assert "Illegal SNPs description" in str(e.value)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["tiny_clean", "tiny_noisy"])
def test_golden_records(ctx, tmp_path, name):
    from golden_util import load_set
    from abawaca_b200 import pipeline
    mg = load_set(name)["mg"]
    paths = synth.write_reference_inputs(mg, str(tmp_path))
    p = pipeline.SamParser(ctx, mg.names)
    for j in range(len(mg.reads)):
        want = p.parse_to_host(open(paths["sams"][j], "rb").read())
        for aligned in (True, False):
            path = str(tmp_path / f"s{j}.bam")
            synth.write_bam(path, mg, j, aligned=aligned, level=6)
            assert np.array_equal(feed_all(ctx, mg.names, open(path, "rb").read(), 1 << 20), want)
    p.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["tiny_clean", "tiny_noisy"])
def test_command_lines_on_bam(tmp_path, name):
    """abawaca-build on BAM samples writes the committed .lrn/.names/.info, and abawaca the committed bins and log"""
    import re
    from golden_util import load_set
    subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "abawaca_b200", "host")], check=True)
    g = load_set(name)
    wd = str(tmp_path)
    paths = synth.write_reference_inputs(g["mg"], wd)
    bams = []
    for j in range(len(g["mg"].reads)):
        bams.append(synth.write_bam(os.path.join(wd, f"sample{j:02d}.bam"), g["mg"], j, aligned=bool(j % 2)))
    outs = {}
    for kind, files in (("bam", bams), ("sam", paths["sams"])):
        build = os.path.join(wd, "build_" + kind)
        r = subprocess.run([os.path.join(BIN, "abawaca-build"), "-f", paths["fasta"], "-o", build, "-s", os.path.join(wd, f"sample*.{kind}"), "-c", files[0]],
                           capture_output=True, text=True)
        assert r.returncode == 0, r.stderr[-2000:]
        outs[kind] = {f: open(os.path.join(build, f)).read() for f in ("abawaca.lrn", "abawaca.names", "abawaca.info")}
    strip = lambda t: "\n".join(l if i != 3 else re.sub(r"sample(\d+)\.(bam|sam)", r"sample\1", l) for i, l in enumerate(t.split("\n")))   # noqa: E731
    assert outs["bam"]["abawaca.lrn"].split("\n")[3] != outs["sam"]["abawaca.lrn"].split("\n")[3]
    for f in outs["bam"]:
        assert strip(outs["bam"][f]) == strip(outs["sam"][f]), f
    lrn = outs["bam"]["abawaca.lrn"].split("\n")
    lrn[3] = "\t".join(os.path.basename(x) for x in lrn[3].split("\t"))
    ref = g["lrn_text"].split("\n")
    ref[3] = "\t".join(os.path.basename(x) for x in ref[3].split("\t"))
    assert strip("\n".join(lrn)) == strip("\n".join(ref))
    assert outs["bam"]["abawaca.names"] == g["names_text"] and outs["bam"]["abawaca.info"] == g["info_text"]
    out = os.path.join(wd, "out")
    env = dict(os.environ, ABW_SCG_LIST=paths["scg_list"])
    r = subprocess.run([os.path.join(BIN, "abawaca"), "-u", os.path.join(wd, "build_bam"), "-o", out, "-c", paths["gene2scg"], "-p", "8"], capture_output=True,
                       text=True, env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    meta = g["meta"]
    assert open(os.path.join(out, "scaf2cluster.txt")).read() == meta["scaf2cluster"]
    assert open(os.path.join(out, "summary.txt")).read() == meta["summary"]
    log = [l.split("]", 1)[1].strip() for l in open(os.path.join(out, "log")) if "Best separation" in l]
    norm = lambda s: re.sub(r"\(\S*/(sample\d+)\.(sam|bam)\)", r"(\1)", s)     # noqa: E731
    assert [norm(x) for x in log] == [norm(x) for x in meta["best_separation_log"]]


@pytest.mark.gpu
def test_large_header(ctx):
    """A header of a million references (an @SQ line for each in the text, and more text) that spans two 64 MB batches: read in time linear in its
    size (the header prefix fetched for parsing grows geometrically), and the records' refIDs resolve through it."""
    import time
    nref = 1_000_000
    refs = [f"contig_{i:07d}" for i in range(nref)]
    lens = [1000 + i % 5000 for i in range(nref)]
    text = "@HD\tVN:1.6\tSO:unsorted\n" + "".join(f"@SQ\tSN:{n}\tLN:{ln}\n" for n, ln in zip(refs, lens)) + "@CO\t" + "x" * (40 << 20) + "\n"
    hdr = synth.bam_header(refs, lens, text=text)
    assert len(hdr) > 64 << 20
    md = _aux("MD", "Z", "50")
    recs = b"".join(synth.bam_record(r, 7 * k, f"q{k}", 0, [(0, 50)], "ACGT" * 12 + "AC", None, md)
                    for k, r in enumerate([0, 1, nref - 1, 424242, -1, 999_998]))
    data = bgzf_file(cut_stream(hdr + recs, [0xff00]), level=1)
    names = [refs[0], refs[424242], refs[nref - 1]]               # a few of them are scaffolds of the assembly
    t0 = time.perf_counter()
    got = feed_all(ctx, names, data, 64 << 20)
    dt = time.perf_counter() - t0
    assert got["scaf"].tolist() == [0, 0xFFFFFFFF, 2, 1, 0xFFFFFFFF, 0xFFFFFFFF]
    assert got["pos0"].tolist() == [0, 7, 14, 21, 28, 35]
    assert dt < 20, dt                                            # a quadratic header walk takes minutes here


def _one_record_file(edit):
    """a BAM file with two records, the second one changed by edit(bytearray of the record) and the file cut inside it"""
    md = _aux("MD", "Z", "50")
    r1 = synth.bam_record(0, 5, "ok", 0, [(0, 50)], "ACGT" * 12 + "AC", None, md)
    r2 = bytearray(synth.bam_record(0, 6, "edited", 0, [(0, 50)], "ACGT" * 12 + "AC", None, md))
    edit(r2)
    return synth.bam_header(EDGE_REFS, EDGE_LENS) + r1 + bytes(r2[:40])


@pytest.mark.gpu
@pytest.mark.parametrize("what", ["block_size_not_int32", "block_size_small", "refid", "l_seq"])
def test_unfinished_record_checked_when_its_fixed_fields_arrive(ctx, what):
    """an unfinished record whose fixed fields are already malformed fails the feed that brings them, not the end of the file; the reader then
    refuses further input"""
    from abawaca_b200 import capi, pipeline
    edit = {"block_size_not_int32": lambda r: r.__setitem__(slice(0, 4), struct.pack("<I", 0x80000000)),
            "block_size_small": lambda r: r.__setitem__(slice(0, 4), struct.pack("<I", 31)),
            "refid": lambda r: r.__setitem__(slice(4, 8), struct.pack("<i", len(EDGE_REFS))),
            "l_seq": lambda r: r.__setitem__(slice(20, 24), struct.pack("<i", 1 << 30))}[what]
    good = bgzf_file([_one_record_file(lambda r: None)], eof=False)
    bad = bgzf_file([_one_record_file(edit)], eof=False)
    r = pipeline.BamReader(ctx, ["chrA"])
    try:
        r.feed(good)                                               # the unfinished second record is carried
        with pytest.raises(capi.AbwError):
            r.finish()
    finally:
        r.close()
    r = pipeline.BamReader(ctx, ["chrA"])
    try:
        with pytest.raises(capi.AbwError, match="status 2"):
            r.feed(bad)
        with pytest.raises(capi.AbwError, match="failed on earlier input"):
            r.feed(synth.BGZF_EOF)
        with pytest.raises(capi.AbwError, match="failed on earlier input"):
            r.finish()
    finally:
        r.close()
