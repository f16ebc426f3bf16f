"""GPU tests of the drop-in command lines: abawaca_b200/bin/abawaca-build and abawaca_b200/bin/abawaca must write the same
files as the reference binaries did when tests/golden/make_golden.py ran them (byte for byte, apart from paths and time stamps)."""
import os
import re
import subprocess

import pytest

from golden_util import load_set

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "abawaca_b200", "bin")


def _norm_lrn(text):
    lines = text.split("\n")
    lines[3] = "\t".join(os.path.basename(x) for x in lines[3].split("\t"))   # the SAM paths in the header differ by directory
    return "\n".join(lines)


@pytest.mark.parametrize("name", ["tiny_clean", "tiny_noisy"])
def test_command_lines_reproduce_reference_files(tmp_path, name, oracle):
    from abawaca_b200 import hostio, synth
    subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "abawaca_b200", "host")], check=True)
    g = load_set(name)
    wd = str(tmp_path)
    paths = synth.write_reference_inputs(g["mg"], wd)
    build = os.path.join(wd, "build")
    r = subprocess.run([os.path.join(BIN, "abawaca-build"), "-f", paths["fasta"], "-o", build, "-s", os.path.join(wd, "sample*.sam"), "-c", paths["sams"][0]],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-2000:]
    assert _norm_lrn(open(os.path.join(build, "abawaca.lrn")).read()) == _norm_lrn(g["lrn_text"])
    assert open(os.path.join(build, "abawaca.names")).read() == g["names_text"]
    assert open(os.path.join(build, "abawaca.info")).read() == g["info_text"]
    assert os.path.exists(os.path.join(build, "abawaca.links")) and os.path.exists(os.path.join(build, "data.txt"))

    out = os.path.join(wd, "out")
    env = dict(os.environ, ABW_SCG_LIST=paths["scg_list"])
    r = subprocess.run([os.path.join(BIN, "abawaca"), "-u", build, "-o", out, "-c", paths["gene2scg"], "-p", "8"], capture_output=True, text=True, env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    meta = g["meta"]
    assert open(os.path.join(out, "scaf2cluster.txt")).read() == meta["scaf2cluster"]
    assert open(os.path.join(out, "summary.txt")).read() == meta["summary"]
    log = [l.split("]", 1)[1].strip() for l in open(os.path.join(out, "log")) if "Best separation" in l]
    strip = lambda s: re.sub(r"\(\S*/(sample\d+\.sam)\)", r"(\1)", s)     # noqa: E731
    assert [strip(x) for x in log] == [strip(x) for x in meta["best_separation_log"]]
    # every final bin has its FASTA, every child cluster its three files
    bins = sorted(set(int(l.split("\t")[1]) for l in meta["scaf2cluster"].splitlines()) - {0})
    for b in bins:
        assert os.path.getsize(os.path.join(out, "final-clusters", f"{b}.fasta")) > 0
    nsplits = len(meta["best_separation_log"])
    for cid in range(2, 2 + 2 * nsplits):
        for ext in ("lrn", "scaf-stats.txt", "scaf-cluster.txt"):
            assert os.path.exists(os.path.join(out, "clusters", f"{cid}.{ext}"))
    # dp2cluster.txt keeps the reference's spurious row for datapoint 0 (quirk Q10)
    assert open(os.path.join(out, "dp2cluster.txt")).readline() == "0\t0\n"
    # the SCG tallies of every child cluster in the log: the oracle's over the scaffolds of <id>.scaf-cluster.txt, printed as std::ostream prints
    # a uint32_t and a double
    prob = hostio.load_search_problem(os.path.join(build, "abawaca.names"), os.path.join(build, "abawaca.lrn"), paths["fasta"], paths["gene2scg"])
    search = oracle.Search(prob["values"], prob["dp2scaf"], prob["T"], prob["len"], prob["scgmask"])
    scaf_id = {s: i for i, s in enumerate(prob["scaf_names"])}
    child_lines = [(int(m.group(1)), m.group(0)) for m in re.finditer(r"Cluster (\d+), \d+ datapoints, \d+ unique SCGs \(\S+ copies\)", open(os.path.join(out, "log")).read())]
    assert sorted(cid for cid, _ in child_lines) == list(range(2, 2 + 2 * nsplits))
    for cid, line in child_lines:
        with open(os.path.join(out, "clusters", f"{cid}.scaf-cluster.txt")) as f:
            scafs = [scaf_id[l.split("\t")[0]] for l in f.read().splitlines()]
        with open(os.path.join(out, "clusters", f"{cid}.lrn")) as f:
            ndps = int(f.readline().split()[1])
        u, avg = search.cluster_scg(scafs)
        assert line == f"Cluster {cid}, {ndps} datapoints, {u} unique SCGs ({avg:g} copies)"
