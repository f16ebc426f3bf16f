"""CPU test: every kernel of the built library starts by waiting for the grid before it (griddepcontrol.wait, ACQBULK in sm_100a SASS).

The library launches its kernels with programmatic stream serialization (csrc/common.cuh, abw_launch_pdl): a grid may be launched while the previous one
still runs, and only the wait keeps it from reading that grid's results early.  One kernel without the wait would also let the grid after it overlap
the grid before it.  The persistent look-back kernels also let their dependents launch (griddepcontrol.launch_dependents, PREEXIT) once their CTAs
leave the ticket loop."""
import os
import re
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "abawaca_b200", "csrc")
LIB = os.path.join(ROOT, "abawaca_b200", "libabawaca_b200.so")
TRIGGERING = ("k_flip_prefix", "k_sweep_ss", "k_sweep_split_scafs", "k_partition2", "k_scan_onepass")


def _cuobjdump():
    for c in (shutil.which("cuobjdump"), os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "cuobjdump")):
        if c and os.path.exists(c):
            return c
    pytest.fail("cuobjdump not found (CUDA toolkit bin directory)")


@pytest.fixture(scope="module")
def sass():
    """mangled kernel name -> its SASS text"""
    subprocess.run(["make", "-s", "-C", CSRC], check=True)
    out = subprocess.run([_cuobjdump(), "-sass", LIB], check=True, capture_output=True, text=True).stdout
    funcs = {}
    name = None
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            name = m.group(1)
            funcs[name] = []
        elif name is not None:
            funcs[name].append(line)
    return {k: "\n".join(v) for k, v in funcs.items()}


def _kernel_names_in_source():
    names = set()
    for f in os.listdir(CSRC):
        if f.endswith((".cu", ".cuh")):
            text = open(os.path.join(CSRC, f)).read()
            names.update(re.findall(r"__global__\s+void\s+(?:__launch_bounds__\([^)]*\)\s*)?(\w+)\s*\(", text))
    return names


def _mangled(name):
    """<length><identifier>, as the identifier appears in an Itanium-mangled name"""
    return str(len(name)) + name


def test_every_kernel_waits_for_the_previous_grid(sass):
    assert sass, "no kernels found in the library"
    missing = sorted(k for k, text in sass.items() if "ACQBULK" not in text)
    assert missing == []


def test_every_kernel_of_the_sources_is_in_the_library(sass):
    src = _kernel_names_in_source()
    assert len(src) >= 60
    assert sorted(n for n in src if not any(_mangled(n) in k for k in sass)) == []


def test_persistent_kernels_trigger_their_dependents(sass):
    for kernel in TRIGGERING:
        texts = [t for k, t in sass.items() if _mangled(kernel) in k]
        assert texts, kernel
        assert all("PREEXIT" in t for t in texts), kernel
