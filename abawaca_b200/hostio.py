"""Python mirror of the on-disk formats at the boundary (SURVEY.md Appendix A).

The product's host side is C++ (abawaca_b200/host/); this module exists so that the Python
tests and bench.py can move the same data between the reference's files and the flat arrays
the C ABI takes.  Format facts cite the reference writer/reader lines.
"""
from __future__ import annotations

import numpy as np

KMER_DIMS = 180


def kmer_dim_names():
    """The 180 canonical 1..4-mer dimension names in .lrn order (abawaca-build.cpp:75-100)."""
    comp = {"A": "T", "C": "G", "G": "C", "T": "A"}
    names, seen = [], {}
    for k in range(1, 5):
        for code in range(4 ** k):
            mer = "".join("ACGT"[(code >> (2 * (k - 1 - i))) & 3] for i in range(k))
            rc = "".join(comp[c] for c in reversed(mer))
            if rc in seen:
                seen[mer] = seen[rc]
            else:
                seen[mer] = len(names)
                names.append(mer)
    return names


def read_fasta(path):
    """SeqIORead_fasta.h:51-103: id = first token after '>', lines trimmed and concatenated."""
    names, seqs, cur = [], [], None
    with open(path, "rb") as f:
        for line in f:
            line = line.strip()
            if not line:
                continue
            if line.startswith(b">"):
                names.append(line[1:].split()[0].decode())
                cur = []
                seqs.append(cur)
            elif cur is not None:
                cur.append(line)
    return names, [b"".join(s) for s in seqs]


def _blocks(mask):
    """(starts, sizes) of the maximal runs of True in a bool array"""
    d = np.diff(np.concatenate(([0], mask.view(np.int8), [0])))
    starts = np.flatnonzero(d == 1)
    return starts.astype(np.uint32), (np.flatnonzero(d == -1) - starts).astype(np.uint32)


def write_twobit(path, names, seqs, version=0, big_endian=False):
    """A UCSC .2bit file of the sequences (bytes), as faToTwoBit writes one: A/C/G/T of either case packed 2 bits per base (T=0 C=1 A=2 G=3, first
    base in the high bits), every other character an N block (the format cannot carry IUPAC codes), lower-case letters mask blocks.
    version 1 has 64-bit record offsets; big_endian writes every word byte-swapped."""
    e = ">" if big_endian else "<"
    code = np.zeros(256, dtype=np.uint8)
    is_acgt = np.zeros(256, dtype=bool)
    for i, c in enumerate(b"TCAG"):
        code[c] = code[c | 0x20] = i
        is_acgt[c] = is_acgt[c | 0x20] = True
    records = []
    for s in seqs:
        a = np.frombuffer(s, dtype=np.uint8)
        ns, nz = _blocks(~is_acgt[a])
        ms, mz = _blocks((a >= ord("a")) & (a <= ord("z")))
        c = code[a]
        c = np.concatenate((c, np.zeros((-c.size) % 4, dtype=np.uint8))).reshape(-1, 4)
        dna = ((c[:, 0] << 6) | (c[:, 1] << 4) | (c[:, 2] << 2) | c[:, 3]).astype(np.uint8).tobytes()
        u32 = lambda x: np.asarray(x, dtype=e + "u4").tobytes()       # noqa: E731
        records.append(u32([a.size, ns.size]) + u32(ns) + u32(nz) + u32([ms.size]) + u32(ms) + u32(mz) + u32([0]) + dna)
    osz = 8 if version else 4
    index_size = sum(1 + len(n.encode()) + osz for n in names)
    off = 16 + index_size
    with open(path, "wb") as f:
        f.write(np.asarray([0x1A412743, version, len(names), 0], dtype=e + "u4").tobytes())
        for n, r in zip(names, records):
            nb = n.encode()
            f.write(bytes([len(nb)]) + nb + np.asarray([off], dtype=e + ("u8" if version else "u4")).tobytes())
            off += len(r)
        for r in records:
            f.write(r)


def write_lrn(path, rows, sample_names, dp_names=None):
    """abawaca-build.cpp:579-606. rows: [ndps][179 + nsamples] truncated values."""
    ndps, ncols = rows.shape
    heads = [n for n in kmer_dim_names() if n != "A"] + list(sample_names)
    assert len(heads) == ncols
    with open(path, "w") as f:
        f.write(f"% {ndps}\n")
        f.write(f"% {ncols + 1}\n")
        f.write("% 9" + "\t1" * ncols + "\n")
        f.write("% Key" + "".join("\t" + h for h in heads) + "\n")
        for i in range(ndps):
            name = (i + 1) if dp_names is None else dp_names[i]
            f.write(str(name) + "".join("\t%.3f" % v for v in rows[i]) + "\n")


def write_names(path, scaf_names, seg_scaf, seg_start, seg_end, seg_nonN):
    """abawaca-build.cpp:578,599 with the segment naming of :217-219."""
    with open(path, "w") as f:
        f.write(f"% {len(seg_scaf)}\n")
        k_in_scaf = {}
        for i in range(len(seg_scaf)):
            s = int(seg_scaf[i])
            k_in_scaf[s] = k_in_scaf.get(s, 0) + 1
            nm = scaf_names[s]
            ln = int(seg_end[i]) - int(seg_start[i]) + 1
            f.write(f"{i + 1}\t{nm}_{k_in_scaf[s]}\t{nm}:({int(seg_start[i])}, {int(seg_end[i])}), {int(seg_nonN[i])}/{ln} non-Ns bps\n")


def write_info(path, scaf_names, lengths, cvg, gc, Ns):
    """abawaca-build.cpp:597"""
    with open(path, "w") as f:
        for i, nm in enumerate(scaf_names):
            f.write("%s\t%d\t%.3f\t%.3f\t%d\n" % (nm, int(lengths[i]), cvg[i], gc[i], int(Ns[i])))


def read_lrn(path):
    """ClusterData.cpp:27-168 -> (dimension names, dp names [n], values [n][D])."""
    with open(path) as f:
        ndps = int(f.readline().split()[1])
        ncols = int(f.readline().split()[1]) - 1
        f.readline()
        heads = f.readline().rstrip("\n").split("\t")[1:]
        assert len(heads) == ncols
        names = np.zeros(ndps, dtype=np.int64)
        vals = np.zeros((ndps, ncols), dtype=np.float64)
        i = 0
        for line in f:
            line = line.rstrip()
            if not line or line[0] == "%":
                continue
            parts = line.split("\t")
            names[i] = int(parts[0])
            vals[i] = [float(x) for x in parts[1:]]   # atof, ClusterData.cpp:159
            i += 1
        assert i == ndps
    return heads, names, vals


def read_names(path):
    """ScafDpData.cpp:41-87 -> list of (dp name, scaffold, start, end, nonN, length)."""
    out = []
    with open(path) as f:
        f.readline()
        for line in f:
            dp, _seg, desc = line.rstrip("\n").split("\t")
            scaf, rest = desc.split(":(", 1)
            coords, tail = rest.split("), ", 1)
            st, en = [int(x) for x in coords.split(", ")]
            nonN, ln = [int(x) for x in tail.split(" ")[0].split("/")]
            out.append((int(dp), scaf, st, en, nonN, ln))
    return out


def load_search_problem(names_path, lrn_path, fasta_path, gene2scg_path=None):
    """Flat arrays of the split-search problem exactly as ScafDpData/ClusterData/SCGdb build them.

    * scaffolds with exactly one dp are dropped (ScafDpData.cpp:92-93, quirk Q1);
    * scaffold ids follow byte-wise name order, dp ids follow (scaffold, dp name) order (:91-99);
    * SCG sets per scaffold, one bit per SCG name (SCGdb.cpp:86-117).
    Returns a dict: values [D][N] (column major), dp2scaf, T, len, scgmask, scaf_names, dp_names, dim_names.
    """
    recs = read_names(names_path)
    by_scaf = {}
    for dp, scaf, st, en, nonN, ln in recs:
        by_scaf.setdefault(scaf, []).append(dp)
    scaf_names = sorted((s for s, d in by_scaf.items() if len(set(d)) != 1), key=lambda s: s.encode())
    dp_names, dp2scaf, T = [], [], []
    for si, s in enumerate(scaf_names):
        d = sorted(set(by_scaf[s]))
        T.append(len(d))
        for x in d:
            dp_names.append(x)
            dp2scaf.append(si)
    heads, lrn_names, vals = read_lrn(lrn_path)
    row_of = {int(n): i for i, n in enumerate(lrn_names)}
    idx = np.array([row_of[x] for x in dp_names], dtype=np.int64)
    values = np.ascontiguousarray(vals[idx].T)
    fa_names, fa_seqs = read_fasta(fasta_path)
    flen = {n: len(s) for n, s in zip(fa_names, fa_seqs)}
    length = np.array([flen[s] for s in scaf_names], dtype=np.uint64)
    sidx = {s: i for i, s in enumerate(scaf_names)}
    scg_of = {}
    scg_names = []
    if gene2scg_path:
        with open(gene2scg_path) as f:
            toks = f.read().split()
        for gene, scg in zip(toks[0::2], toks[1::2]):
            scaf = gene[:gene.rfind("_")]
            if scaf in sidx:
                scg_of.setdefault(sidx[scaf], set()).add(scg)
        scg_names = sorted({g for v in scg_of.values() for g in v})
    gi = {g: i for i, g in enumerate(scg_names)}
    W = max(1, (len(scg_names) + 63) // 64)
    mask = np.zeros((len(scaf_names), W), dtype=np.uint64)
    for s, gs in scg_of.items():
        for g in gs:
            mask[s, gi[g] // 64] |= np.uint64(1) << np.uint64(gi[g] % 64)
    return dict(values=values, dp2scaf=np.array(dp2scaf, dtype=np.uint32), T=np.array(T, dtype=np.uint32), len=length,
                scgmask=mask, scaf_names=scaf_names, dp_names=np.array(dp_names, dtype=np.int64), dim_names=heads)
