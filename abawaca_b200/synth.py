"""Seeded synthetic metagenomes for the abawaca hot path (SURVEY.md section 8d).

There is no network, so every workload is synthetic: scaffolds drawn from
synthetic genomes with genome-specific oligonucleotide composition, synthetic
per-sample coverage (read records), and synthetic single-copy-gene (SCG)
placements.  The same object can be

  * handed to the CUDA path / the flat-array oracle as flat numpy arrays, or
  * written as the text files the reference binaries read (FASTA, SAM,
    gene2scg, scg.list) -- see `write_reference_inputs`.

Scaffolds are emitted in byte-wise name order, because both reference programs
order scaffolds through `std::map<std::string, ...>`
(abawaca-build.cpp:482,596; ScafDpData.cpp:59,91).
"""
from __future__ import annotations

import dataclasses
import os
import struct
import zlib
from concurrent.futures import ThreadPoolExecutor

import numpy as np

MASTER_SEED = 20261018
READ_DTYPE = np.dtype([("scaf", "<u4"), ("pos0", "<u4"), ("len", "<u4"), ("flag_nsnps", "<u4")])

_TRIMERS = np.array([[ord("ACGT"[(t >> 4) & 3]), ord("ACGT"[(t >> 2) & 3]), ord("ACGT"[t & 3])] for t in range(64)], dtype=np.uint8)


@dataclasses.dataclass
class Metagenome:
    names: list            # scaffold names, byte-wise sorted
    genome: np.ndarray     # [S] genome of each scaffold
    offsets: np.ndarray    # [S+1] uint64 offsets into `seq`
    seq: np.ndarray        # uint8 ASCII, concatenated scaffolds
    reads: list            # per sample: structured array READ_DTYPE, in "SAM order"
    scg_names: list        # the SCG vocabulary (scg.list)
    gene2scg: list         # (gene name "<scaf>_<idx>", scg name)
    read_len: int
    seed: int

    @property
    def nscaf(self):
        return len(self.names)

    def scaffold(self, i):
        return self.seq[int(self.offsets[i]):int(self.offsets[i + 1])]

    def scg_masks(self, scaf_index_of_name=None):
        """uint64 [S][W] bit masks of SCG names per scaffold (sets, SCGdb.h:25)."""
        idx = {n: i for i, n in enumerate(self.names)} if scaf_index_of_name is None else scaf_index_of_name
        gidx = {n: i for i, n in enumerate(sorted(set(s for _, s in self.gene2scg)))}
        W = max(1, (len(gidx) + 63) // 64)
        masks = np.zeros((len(idx), W), dtype=np.uint64)
        for gene, scg in self.gene2scg:
            scaf = gene[:gene.rfind("_")]
            if scaf in idx:
                g = gidx[scg]
                masks[idx[scaf], g // 64] |= np.uint64(1) << np.uint64(g % 64)
        return masks


def make_metagenome(n_scaffolds, n_samples, n_genomes, seed, *, min_len=4000, mean_extra=6000, max_len=200000,
                    read_len=150, cov_lo=0.5, cov_hi=16.0, n_run_frac=0.005, n_scg=51, scg_p=0.9,
                    bad_read_frac=0.03, q6_reads=False, shuffle_reads=False, with_reads=True,
                    gc_lo=0.25, gc_hi=0.75, tri_sigma=0.6, shard=None, bimodal_frac=0.0, bimodal_factor=4.0) -> Metagenome:
    """shard: when given, the genome models (composition, coverage) still come from `seed` alone, but the scaffolds, reads and gene
    placements are drawn from (seed, shard): several shards are then pieces of ONE community, which is how bench.py builds the
    N-GPU workload (every rank generates only its own scaffolds).
    bimodal_frac: that share of the genomes gets two coverage modes (half of their scaffolds are covered bimodal_factor times deeper in every
    sample) while their single-copy genes stay spread over all their scaffolds: a clean separation INSIDE one genome, which only the SCG test of
    ClusterQuality::is_split_better (disjoint SCG sets on the two sides) turns down.  Drawn from its own generator: 0 leaves every other set as it was."""
    rng = np.random.default_rng(seed)
    # genome models
    gc = rng.uniform(gc_lo, gc_hi, n_genomes)
    base_p = np.stack([(1 - gc) / 2, gc / 2, gc / 2, (1 - gc) / 2], axis=1)  # A C G T
    tri_p = np.empty((n_genomes, 64))
    for t in range(64):
        tri_p[:, t] = base_p[:, (t >> 4) & 3] * base_p[:, (t >> 2) & 3] * base_p[:, t & 3]
    tri_p *= np.exp(rng.normal(0.0, tri_sigma, (n_genomes, 64)))
    tri_p /= tri_p.sum(axis=1, keepdims=True)
    cov = np.exp(rng.uniform(np.log(cov_lo), np.log(cov_hi), (n_genomes, max(n_samples, 1))))
    tag = ""
    if shard is not None:
        rng = np.random.default_rng([seed, 7919 + int(shard)])
        tag = f"r{int(shard)}_"

    genome = rng.integers(0, n_genomes, n_scaffolds)
    lengths = np.minimum(min_len + rng.exponential(mean_extra, n_scaffolds).astype(np.int64), max_len)
    names = [f"{tag}g{g}_scaffold_{i}" for i, g in enumerate(genome)]
    order = sorted(range(n_scaffolds), key=lambda i: names[i].encode())
    names = [names[i] for i in order]
    genome = genome[order]
    lengths = lengths[order]
    offsets = np.zeros(n_scaffolds + 1, dtype=np.uint64)
    offsets[1:] = np.cumsum(lengths)
    seq = np.empty(int(offsets[-1]), dtype=np.uint8)
    ntri = (lengths + 2) // 3
    for g in range(n_genomes):
        idx = np.nonzero(genome == g)[0]
        if idx.size == 0:
            continue
        total = int(ntri[idx].sum())
        tri = rng.choice(64, size=total, p=tri_p[g]).astype(np.uint8)
        bases = _TRIMERS[tri].reshape(-1)
        o = 0
        for i in idx:
            L = int(lengths[i])
            seq[int(offsets[i]):int(offsets[i]) + L] = bases[o:o + L]
            o += int(ntri[i]) * 3
    # a few runs of N
    n_with_n = int(round(n_run_frac * n_scaffolds))
    if n_with_n > 0:
        for i in rng.choice(n_scaffolds, size=n_with_n, replace=False):
            L = int(lengths[i])
            run = int(rng.integers(10, 101))
            p = int(rng.integers(0, L - run))
            seq[int(offsets[i]) + p:int(offsets[i]) + p + run] = ord("N")

    cov_mult = np.ones(n_scaffolds)
    if bimodal_frac > 0:
        rng2 = np.random.default_rng([seed, 424243] + ([int(shard)] if shard is not None else []))
        bimodal = rng2.random(n_genomes) < bimodal_frac
        deep = rng2.random(n_scaffolds) < 0.5
        cov_mult = np.where(bimodal[genome] & deep, bimodal_factor, 1.0)
    # reads, one record stream per sample, scaffold-major with random positions
    reads = []
    if with_reads:
        for j in range(n_samples):
            lam = cov[genome, j] * cov_mult * lengths / read_len
            n = np.floor(lam + rng.random(n_scaffolds)).astype(np.int64)
            if q6_reads and j == n_samples - 1:
                extra = (lengths + 999) // 1000
            else:
                extra = np.zeros(n_scaffolds, dtype=np.int64)
            tot = n + extra
            rec = np.zeros(int(tot.sum()), dtype=READ_DTYPE)
            scaf_of = np.repeat(np.arange(n_scaffolds, dtype=np.uint32), tot)
            start_of = np.repeat(np.cumsum(tot) - tot, tot)
            k = np.arange(rec.size) - start_of           # index of the read within its scaffold
            L_of = lengths[scaf_of]
            n_of = n[scaf_of]
            span = np.maximum(L_of - read_len, 0) + 1
            pos = (rng.random(rec.size) * span).astype(np.int64)
            is_extra = k >= n_of
            pos = np.where(is_extra, np.minimum((k - n_of) * 1000, np.maximum(L_of - read_len, 0)), pos)
            flag = np.zeros(rec.size, dtype=np.uint32)
            nsnps = np.zeros(rec.size, dtype=np.uint32)
            if bad_read_frac > 0:
                u = rng.random(rec.size)
                b = bad_read_frac / 3
                flag = np.where((u < b) & ~is_extra, 0x100, flag)            # secondary alignment
                flag = np.where((u >= b) & (u < 2 * b) & ~is_extra, 0x4, flag)  # unmapped
                nsnps = np.where((u >= 2 * b) & (u < 3 * b) & ~is_extra, 16, nsnps)
                nsnps = np.where((u >= 3 * b) & (u < 4 * b), 3, nsnps)     # a few tolerated mismatches
            rec["scaf"] = scaf_of
            rec["pos0"] = pos.astype(np.uint32)
            rec["len"] = read_len
            rec["flag_nsnps"] = (flag & 0xFFFF) | (nsnps.astype(np.uint32) << 16)
            if shuffle_reads:
                rec = rec[rng.permutation(rec.size)]
            reads.append(rec)

    # single-copy genes
    scg_names = [f"SCG{i + 1:02d}" for i in range(n_scg)]
    gene2scg = []
    gene_counter = {}
    for g in range(n_genomes):
        idx = np.nonzero(genome == g)[0]
        if idx.size == 0:
            continue
        for s in range(n_scg):
            if rng.random() < scg_p:
                i = int(idx[rng.integers(0, idx.size)])
                gene_counter[i] = gene_counter.get(i, 0) + 1
                gene2scg.append((f"{names[i]}_{gene_counter[i]}", scg_names[s]))
    return Metagenome(names, genome, offsets, seq, reads, scg_names, gene2scg, read_len, seed)


CONFIGS = {
    # BASELINE.json configs -> generator arguments (SURVEY.md section 8d)
    "cfg1": dict(n_scaffolds=2000, n_samples=3, n_genomes=8, seed=MASTER_SEED + 1),
    "cfg2": dict(n_scaffolds=50000, n_samples=10, n_genomes=32, seed=MASTER_SEED + 2),
    "cfg3": dict(n_scaffolds=500000, n_samples=20, n_genomes=128, seed=MASTER_SEED + 3),
    "cfg4": dict(n_scaffolds=1000000, n_samples=50, n_genomes=256, seed=MASTER_SEED + 4),
}


def write_reference_inputs(mg: Metagenome, directory: str):
    """Write FASTA + one SAM per sample + gene2scg + scg.list, the text inputs of the reference binaries.

    SAM lines have the >= 11 tab fields `ReadMapping(const char*)` needs
    (ReadMapping.cpp:36-69).  Mismatches are encoded in MD:Z so that
    `num_snps()` equals the record's nsnps.
    """
    os.makedirs(directory, exist_ok=True)
    fa = os.path.join(directory, "assembly.fa")
    with open(fa, "w") as f:
        for i, name in enumerate(mg.names):
            s = mg.scaffold(i).tobytes().decode()
            f.write(f">{name}\n")
            for o in range(0, len(s), 80):
                f.write(s[o:o + 80] + "\n")
    sams = []
    for j, rec in enumerate(mg.reads):
        path = os.path.join(directory, f"sample{j:02d}.sam")
        sams.append(path)
        with open(path, "w") as f:
            f.write("@HD\tVN:1.0\tSO:unsorted\n")
            for r, (scaf, pos0, ln, fn) in enumerate(rec.tolist()):
                flag, nsnps = fn & 0xFFFF, fn >> 16
                seq = "A" * ln
                qual = "I" * ln
                if nsnps == 0:
                    md = f"MD:Z:{ln}"
                else:  # nsnps isolated mismatches at the start of the read
                    md = "MD:Z:0" + "".join("C0" for _ in range(nsnps - 1)) + f"C{ln - nsnps}"
                rname = "*" if (flag & 0x4) else mg.names[scaf]
                pos1 = 0 if (flag & 0x4) else pos0 + 1
                cigar = "*" if (flag & 0x4) else f"{ln}M"
                tail = "" if (flag & 0x4) else "\t" + md
                f.write(f"r{j}_{r}/1\t{flag}\t{rname}\t{pos1}\t42\t{cigar}\t*\t0\t0\t{seq}\t{qual}{tail}\n")
    g2s = os.path.join(directory, "genes.scg")
    with open(g2s, "w") as f:
        for gene, scg in mg.gene2scg:
            f.write(f"{gene}\t{scg}\n")
    lst = os.path.join(directory, "scg.list")
    with open(lst, "w") as f:
        for s in mg.scg_names:
            f.write(s + "\n")
    return dict(fasta=fa, sams=sams, gene2scg=g2s, scg_list=lst)


# ---- BAM ------------------------------------------------------------------------------------------------------------------------
BGZF_EOF = bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")
_BAM_FIXED = np.dtype([("block_size", "<i4"), ("refID", "<i4"), ("pos", "<i4"), ("l_read_name", "u1"), ("mapq", "u1"), ("bin", "<u2"),
                       ("n_cigar_op", "<u2"), ("flag", "<u2"), ("l_seq", "<i4"), ("next_refID", "<i4"), ("next_pos", "<i4"), ("tlen", "<i4")])
_NT16 = np.full(256, 15, dtype=np.uint8)
for _i, _c in enumerate("=ACMGRSVTWYHKDBN"):
    _NT16[ord(_c)] = _i
    _NT16[ord(_c.lower())] = _i


def bam_header(names, lengths, text="@HD\tVN:1.6\tSO:unsorted\n") -> bytes:
    """magic, SAM header text and the reference list"""
    out = [b"BAM\1", struct.pack("<i", len(text)), text.encode(), struct.pack("<i", len(names))]
    for n, ln in zip(names, lengths):
        b = n.encode() + b"\0"
        out += [struct.pack("<i", len(b)), b, struct.pack("<i", int(ln))]
    return b"".join(out)


def bam_record(refID, pos, name, flag, cigar=(), seq="", qual=None, aux=b"", mapq=42, next_refID=-1, next_pos=-1, tlen=0) -> bytes:
    """one BAM record; cigar: (op code, length) pairs, seq: the bases as text, aux: the encoded aux fields"""
    nb = name.encode() + b"\0"
    codes = _NT16[np.frombuffer(seq.encode(), dtype=np.uint8)] if seq else np.zeros(0, dtype=np.uint8)
    if codes.size % 2:
        codes = np.append(codes, 0)
    packed = ((codes[0::2] << 4) | codes[1::2]).astype(np.uint8).tobytes()
    q = bytes([0xFF] * len(seq)) if qual is None else bytes(qual)
    body = struct.pack("<iiBBHHHiiii", refID, pos, len(nb), mapq, 4680, len(cigar), flag, len(seq), next_refID, next_pos, tlen) + nb + \
        b"".join(struct.pack("<I", (ln << 4) | op) for op, ln in cigar) + packed + q + aux
    return struct.pack("<i", len(body)) + body


def _md_text(ln, nsnps):
    if nsnps == 0:
        return f"{ln}"
    return "0" + "".join("C0" for _ in range(nsnps - 1)) + f"C{ln - nsnps}"    # as write_reference_inputs writes it


def sample_bam_records(mg: Metagenome, j, seed=0, chunk=1 << 17):
    """The records of sample j as BAM, in chunks: (uint8 array of whole records, record sizes).  The fields are those of the SAM lines
    write_reference_inputs writes (FLAG, RNAME, POS, CIGAR {len}M, the MD:Z field, no fields for unmapped reads), with the scaffold's bases as
    SEQ and random qualities; the read names are zero-padded."""
    rec = mg.reads[j]
    rng = np.random.default_rng([seed, 5813, j])
    nscaf = mg.nscaf
    slen = np.diff(mg.offsets.astype(np.int64))
    for c0 in range(0, rec.size, chunk):
        r = rec[c0:c0 + chunk]
        n = r.size
        flag = (r["flag_nsnps"] & 0xFFFF).astype(np.uint32)
        nsnps = (r["flag_nsnps"] >> 16).astype(np.uint32)
        ln = r["len"].astype(np.int64)
        unm = (flag & 4) != 0
        keys = np.stack([unm.astype(np.int64), nsnps.astype(np.int64), ln], axis=1)
        groups, inv = np.unique(keys, axis=0, return_inverse=True)
        inv = inv.reshape(-1)
        names_w = 9
        prefix = f"r{j}_".encode()
        lrn = len(prefix) + names_w + 3
        size = np.zeros(n, dtype=np.int64)
        parts = []
        for g, (u, ns, L) in enumerate(groups.tolist()):
            sel = np.flatnonzero(inv == g)
            aux = b"" if u else b"MDZ" + _md_text(L, ns).encode() + b"\0"
            ncig = 0 if u else 1
            reclen = 36 + lrn + 4 * ncig + (L + 1) // 2 + L + len(aux)
            size[sel] = reclen
            parts.append((sel, reclen, u, L, aux, ncig))
        off = np.zeros(n + 1, dtype=np.int64)
        off[1:] = np.cumsum(size)
        buf = np.zeros(int(off[-1]), dtype=np.uint8)
        for sel, reclen, u, L, aux, ncig in parts:
            k = sel.size
            rows = np.zeros((k, reclen), dtype=np.uint8)
            fx = np.zeros(k, dtype=_BAM_FIXED)
            fx["block_size"] = reclen - 4
            fx["refID"] = -1 if u else r["scaf"][sel].astype(np.int64)
            fx["pos"] = -1 if u else r["pos0"][sel].astype(np.int64)
            fx["l_read_name"] = lrn
            fx["mapq"] = 42
            fx["bin"] = 4680
            fx["n_cigar_op"] = ncig
            fx["flag"] = flag[sel]
            fx["l_seq"] = L
            fx["next_refID"] = -1
            fx["next_pos"] = -1
            rows[:, :36] = fx.view(np.uint8).reshape(k, 36)
            o = 36
            rows[:, o:o + len(prefix)] = np.frombuffer(prefix, dtype=np.uint8)
            num = (c0 + sel).astype(np.int64)
            for d in range(names_w):
                rows[:, o + len(prefix) + names_w - 1 - d] = 48 + (num // 10 ** d) % 10
            rows[:, o + len(prefix) + names_w:o + lrn] = np.frombuffer(b"/1\0", dtype=np.uint8)
            o += lrn
            if ncig:
                rows[:, o:o + 4] = np.frombuffer(struct.pack("<I", L << 4), dtype=np.uint8)
                o += 4
            sc = np.minimum(r["scaf"][sel].astype(np.int64), nscaf - 1)
            p = np.minimum(r["pos0"][sel].astype(np.int64)[:, None] + np.arange(L), slen[sc][:, None] - 1)
            codes = _NT16[mg.seq[mg.offsets[sc].astype(np.int64)[:, None] + np.maximum(p, 0)]]
            if L % 2:
                codes = np.concatenate([codes, np.zeros((k, 1), dtype=np.uint8)], axis=1)
            rows[:, o:o + (L + 1) // 2] = (codes[:, 0::2] << 4) | codes[:, 1::2]
            o += (L + 1) // 2
            rows[:, o:o + L] = rng.integers(0, 41, (k, L), dtype=np.uint8)
            o += L
            rows[:, o:] = np.frombuffer(aux, dtype=np.uint8)
            buf[(off[sel][:, None] + np.arange(reclen)).reshape(-1)] = rows.reshape(-1)
        yield buf, size


def _bgzf_block(payload, level, strategy) -> bytes:
    c = zlib.compressobj(level, zlib.DEFLATED, -15, 9, strategy)
    cdata = c.compress(payload) + c.flush()
    return struct.pack("<BBBBIBBHBBHH", 31, 139, 8, 4, 0, 0, 255, 6, ord("B"), ord("C"), 2, len(cdata) + 25) + cdata + \
        struct.pack("<II", zlib.crc32(payload), len(payload))


class BgzfWriter:
    """BGZF blocks of a byte stream.  aligned=True cuts as htslib does: a block holds at most 0xff00 bytes and a new block starts before a record
    that would not fit (records longer than that are split); aligned=False cuts wherever the running byte count says, into pieces of `cut` bytes or,
    without it, of random sizes in 1 .. 0xff00 (records and the header then cross blocks, as htsjdk writes them)."""

    def __init__(self, f, aligned=True, level=6, strategy=zlib.Z_DEFAULT_STRATEGY, cut=None, seed=0, threads=8):
        self.f, self.aligned, self.level, self.strategy, self.cut = f, aligned, level, strategy, cut
        self.rng = np.random.default_rng([seed, 4099])
        self.pool = ThreadPoolExecutor(threads)
        self.pend = b""
        self.k = self._piece()

    def _emit(self, payloads):
        for blk in self.pool.map(lambda p: _bgzf_block(p, self.level, self.strategy), payloads):
            self.f.write(blk)

    def _piece(self):
        return self.cut if self.cut else int(self.rng.integers(1, 0xff00 + 1))

    def write(self, data, sizes=None):
        """data: bytes or uint8 array; sizes: the record sizes it consists of (aligned mode), None for one unit (e.g. the header)"""
        data = bytes(data) if not isinstance(data, bytes) else data
        if not self.aligned:
            buf = self.pend + data
            pieces, o = [], 0
            while o + self.k <= len(buf):
                pieces.append(buf[o:o + self.k])
                o += self.k
                self.k = self._piece()
            self.pend = buf[o:]
            self._emit(pieces)
            return
        ends = np.cumsum(np.asarray([len(data)] if sizes is None else sizes, dtype=np.int64))
        starts = ends - np.asarray([len(data)] if sizes is None else sizes, dtype=np.int64)
        pieces, cur, i = [], self.pend, 0
        while i < ends.size:
            room = 0xff00 - len(cur)
            # records i .. j-1 fit into the open block
            j = int(np.searchsorted(ends, starts[i] + room, side="right"))
            if j > i:
                cur += data[starts[i]:ends[j - 1]]
                i = j
                continue
            if cur:
                pieces.append(cur)
                cur = b""
                continue
            rec = data[starts[i]:ends[i]]                      # longer than a block: split
            for o in range(0, len(rec), 0xff00):
                pieces.append(rec[o:o + 0xff00])
            cur = pieces.pop()
            i += 1
        self.pend = cur
        self._emit(pieces)

    def flush(self):
        """end the open block (htslib flushes after the header)"""
        if self.aligned and self.pend:
            self._emit([self.pend])
            self.pend = b""

    def close(self, eof=True):
        if self.pend:
            rest = self.pend
            self.pend = b""
            self._emit([rest[o:o + 0xff00] for o in range(0, len(rest), 0xff00)])
        if eof:
            self.f.write(BGZF_EOF)
        self.pool.shutdown()


def write_bam(path, mg: Metagenome, j, aligned=True, level=6, strategy=zlib.Z_DEFAULT_STRATEGY, cut=None, seed=0, threads=8):
    """Sample j as a BAM file (the reads of write_reference_inputs' SAM file), in htslib's block layout or cut at arbitrary sizes."""
    with open(path, "wb") as f:
        w = BgzfWriter(f, aligned=aligned, level=level, strategy=strategy, cut=cut, seed=seed, threads=threads)
        w.write(bam_header(mg.names, np.diff(mg.offsets.astype(np.int64))))
        w.flush()
        for buf, size in sample_bam_records(mg, j, seed=seed):
            w.write(buf, size)
        w.close()
    return path
