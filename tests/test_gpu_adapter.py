"""GPU test of the drop-in seam: oracle/_ref/ref_search_gpu is the reference's OWN work list and data model (compiled from
/root/reference/src) in which every ClusterSeparator::separate() call is served by ClusterSeparatorGPU, a subclass of the
reference's strategy class that forwards to libabawaca_b200.so (oracle/ref_gpu_adapter.h).  Its dump must be character for
character the dump of the pure reference (the committed golden)."""
import os
import subprocess

import pytest

from golden_util import load_set

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "oracle", "_ref", "ref_search_gpu")


@pytest.mark.skipif(not os.path.exists(EXE), reason="oracle/_ref/ref_search_gpu is built by `make -C oracle ref` only where the reference's C++ sources are present")
@pytest.mark.parametrize("name", ["tiny_clean", "tiny_noisy"])
@pytest.mark.parametrize("strategy", ["sensspec", "splitscafs"])
def test_reference_driver_with_gpu_separator_matches_reference(tmp_path, name, strategy):
    g = load_set(name)
    mg = g["mg"]
    wd = str(tmp_path)
    files = {}
    for key, text in (("names", g["names_text"]), ("lrn", g["lrn_text"]), ("info", g["info_text"])):
        files[key] = os.path.join(wd, key)
        open(files[key], "w").write(text)
    files["fasta"] = os.path.join(wd, "assembly.fa")
    with open(files["fasta"], "w") as f:
        for i, nm in enumerate(mg.names):
            f.write(f">{nm}\n{mg.scaffold(i).tobytes().decode()}\n")
    files["scg"] = os.path.join(wd, "genes.scg")
    open(files["scg"], "w").write("".join(f"{a}\t{b}\n" for a, b in mg.gene2scg))
    files["list"] = os.path.join(wd, "scg.list")
    open(files["list"], "w").write("\n".join(mg.scg_names) + "\n")
    out = os.path.join(wd, "dump.tsv")
    r = subprocess.run([EXE, files["names"], files["fasta"], files["info"], files["lrn"], files["scg"], files["list"], strategy, "4", out],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-2000:]
    assert open(out).read() == g["meta"]["ref_search"][strategy]
