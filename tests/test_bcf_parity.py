"""Whole-file parity of the drop-in binding (SURVEY section 8c / VERDICT r1 item 1): `delly_b200 sr|lr` (bindings/delly_b200_main.cpp: htslib
reads the BAM into record lists, the batched stage mirrors run the chain, htslib writes the BCF) against what the reference's OWN drivers —
src/delly.h + src/tegua.h and every header they include compiled verbatim and linked against the same htslib (oracle/_ref/delly_ref,
oracle/ref_main11.cpp) — wrote for the same command on the reference's own fixtures example/sr.bam, example/lr.bam, example/ref.fa
(oracle/_ref/example, copied at build time). The reference's outputs are stored in tests/golden/bcf_parity.npz (written by
tests/golden/make_bcf_parity.py), so no reference binary runs here. The BCF must be identical byte for byte once the BGZF container is
inflated, the only exception being the ##fileDate header line (src/modvcf.h:360-364); the CSI index must be identical too. Both sides run in
the example directory with relative input names, so the ##reference header line carries no machine path.

[gpu]            the real binary (delly_b200/bin/delly_b200) on a B200: every alignment batch on the device.
[edlib-standin]  the CPU suite: the same binding source compiled with the alignment entry points forwarded to the reference's own
                 functions (tests/standin/binding_standin.cpp) — checks the IO glue, option handling, stage sequence and the BCF writer."""
import gzip
import os
import re
import subprocess

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
REFDIR = os.path.join(ROOT, "oracle", "_ref")
EX = os.path.join(REFDIR, "example")
GOLD = os.path.join(HERE, "golden", "bcf_parity.npz")

# case -> (mode, input BAMs, options); "-x" takes the exclude file of the case (_exclude_lines), "-v" the site list the reference wrote for
# the named discovery case (stored with the golden outputs)
CASES = {
    "sr": ("sr", ["sr.bam"], []),
    "lr": ("lr", ["lr.bam"], []),
    "sr_options": ("sr", ["sr.bam"], ["-t", "DEL,INV", "-q", "10", "-z", "3", "-p", "12", "-c", "30"]),
    "sr_genotyping": ("sr", ["sr.bam"], ["-v", "sr"]),
    "lr_genotyping": ("lr", ["lr.bam"], ["-v", "lr"]),
    "sr_two_samples": ("sr", ["sr.bam", "sr.bam"], []),
    "sr_exclude_discovery": ("sr", ["sr.bam"], ["-x"]),
    "sr_exclude_genotyping": ("sr", ["sr.bam"], ["-x", "-v", "sr"]),
    "lr_exclude": ("lr", ["lr.bam"], ["-x"]),
}
VCF_TEXT_CASE = "sr"       # `-o -`: the VCF text on stdout, stored as "sr.vcf"


def _exclude_lines(case):
    """exclude intervals in the reference's format (src/util.h:666-741: `chr start end` per line, or a bare `chr` for a whole contig)"""
    fai = [l.split("\t") for l in open(os.path.join(EX, "ref.fa.fai"))]
    name, length = fai[0][0], int(fai[0][1])
    if case.startswith("sr"):
        return [f"{name}\t{length // 3}\t{length // 3 + length // 8}", f"{name}\t{length - 2000}\t{length - 500}"]
    return [f"{name}\t{length // 2}\t{length // 2 + length // 10}"]


def case_command(case, out, tmp_path, sites):
    """The command line of a case after the executable, run with cwd=EX; `sites(name)` returns the path of a stored site list."""
    mode, bams, opts = CASES[case]
    args = [mode, "-g", "ref.fa"]
    i = 0
    while i < len(opts):
        if opts[i] == "-x":
            p = os.path.join(str(tmp_path), "exclude.tsv")
            with open(p, "w") as f:
                f.write("".join(line + "\n" for line in _exclude_lines(case)))
            args += ["-x", p]
            i += 1
        elif opts[i] == "-v":
            args += ["-v", sites(opts[i + 1])]
            i += 2
        else:
            args.append(opts[i])
            i += 1
    return args + ["-o", out] + bams


def _standin_binary():
    from oracle import pyoracle
    pyoracle.build()
    out = os.path.join(HERE, "standin", "_build")
    os.makedirs(out, exist_ok=True)
    exe = os.path.join(out, "delly_b200_standin")
    deps = [os.path.join(HERE, "standin", f) for f in ("binding_standin.cpp", "host_standin.cpp")]
    deps += [os.path.join(ROOT, "bindings", f) for f in os.listdir(os.path.join(ROOT, "bindings"))]
    deps += [os.path.join(ROOT, "delly_b200", "host", f) for f in os.listdir(os.path.join(ROOT, "delly_b200", "host"))]
    if not os.path.exists(exe) or os.path.getmtime(exe) < max(os.path.getmtime(f) for f in deps):
        import delly_b200
        delly_b200.lib()
        pkg = os.path.join(ROOT, "delly_b200")
        hts = os.path.join(REFDIR, "hts")      # htslib archive and public headers, built with the checkers (tools/build_htslib.sh)
        r = subprocess.run(["g++", "-std=c++17", "-O2", "-w", "-o", exe, os.path.join(HERE, "standin", "binding_standin.cpp"), "-I" + os.path.join(hts, "include"),
                            "-L" + REFDIR, "-l:libdelly_ref.so", "-L" + pkg, "-l:libdelly_b200.so", "-Wl,-rpath," + REFDIR, "-Wl,-rpath," + pkg,
                            os.path.join(hts, "libhts.a"), "-lz", "-lm", "-lpthread"], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
    return exe


@pytest.fixture(params=[pytest.param("gpu", marks=pytest.mark.gpu), "edlib-standin"])
def binding(request):
    assert os.path.isdir(EX), "oracle/_ref/example missing: __graft_entry__.build() copies the reference's example data there"
    if request.param == "gpu":
        exe = os.path.join(ROOT, "delly_b200", "bin", "delly_b200")
        assert os.path.exists(exe), "delly_b200/bin/delly_b200 not built"
        return [exe]
    return [_standin_binary(), "--mei", os.path.join(ROOT, "delly_b200", "data", "_mei_templates.fa")]


def _inflate(path):
    raw = gzip.open(path, "rb").read()
    return re.sub(rb"##fileDate=\d+\n", b"##fileDate=X\n", raw, count=1)


def _run(cmd, **kw):
    r = subprocess.run(cmd, capture_output=True, text=True, **kw)
    assert r.returncode == 0, (cmd, r.stderr[-2000:])
    return r


@pytest.fixture(scope="module")
def golden():
    with np.load(GOLD) as z:
        return {k: z[k].tobytes() for k in z.files}


def _sites(golden, tmp_path):
    def path(name):
        p = os.path.join(str(tmp_path), name + ".sites.bcf")
        for ext in ("", ".csi"):
            with open(p + ext, "wb") as f:
                f.write(golden[name + ".sites.bcf" + ext])
        return p
    return path


def _pair(binding, golden, case, tmp_path):
    our_out = str(tmp_path / "ours.bcf")
    mei = binding[1:] if CASES[case][0] == "lr" else []
    args = case_command(case, our_out, tmp_path, _sites(golden, tmp_path))
    _run([binding[0], args[0]] + mei + args[1:], cwd=EX)
    a, b = golden[case + ".bcf"], _inflate(our_out)
    assert len(a) > 1000
    assert a == b, "BCF streams differ"
    assert golden[case + ".bcf.csi"] == open(our_out + ".csi", "rb").read()
    return a


def test_example_sr_bcf_identical(binding, golden, tmp_path):
    """`delly sr -g example/ref.fa example/sr.bam` (BASELINE configs[0])"""
    a = _pair(binding, golden, "sr", tmp_path)
    assert b"DEL00000000" in a and b"CONSENSUS" in a


def test_example_lr_bcf_identical(binding, golden, tmp_path):
    """`delly lr -g example/ref.fa example/lr.bam`"""
    a = _pair(binding, golden, "lr", tmp_path)
    assert b"DEL00000000" in a


def test_example_sr_vcf_text_identical(binding, golden):
    """-o - : the VCF text on stdout (src/modvcf.h:355-357)"""
    a = golden[VCF_TEXT_CASE + ".vcf"].decode()
    b = _run([binding[0], "sr", "-g", "ref.fa", "sr.bam"], cwd=EX).stdout
    strip = lambda t: re.sub(r"##fileDate=\d+\n", "", t)
    assert strip(a) == strip(b) and "\tPRECISE;SVTYPE=DEL;" in a


def test_example_sr_options_and_type_restriction(binding, golden, tmp_path):
    """non-default options reach the stages: -t DEL,INV, map-qual, clique size, max-reads"""
    _pair(binding, golden, "sr_options", tmp_path)


def test_example_sr_genotyping_mode_round_trip(binding, golden, tmp_path):
    """`delly sr -v sites.bcf`: the discovery output of the reference genotyped again (BASELINE configs[3] shape)"""
    _pair(binding, golden, "sr_genotyping", tmp_path)


def test_example_lr_genotyping_mode_round_trip(binding, golden, tmp_path):
    _pair(binding, golden, "lr_genotyping", tmp_path)


def test_two_samples_one_call_set(binding, golden, tmp_path):
    """two input files (the same library twice): sample names are made unique, discovery pools the files, one FORMAT column each"""
    a = _pair(binding, golden, "sr_two_samples", tmp_path)
    assert b"sr_0" in a


@pytest.mark.parametrize("mode", ["discovery", "genotyping"])
def test_example_sr_with_exclude_intervals(binding, golden, tmp_path, mode):
    """-x: scan, clustering, assembly and the library estimate run over the valid regions only, the genotyping pass over whole contigs"""
    _pair(binding, golden, "sr_exclude_" + mode, tmp_path)


def test_example_lr_with_exclude_intervals(binding, golden, tmp_path):
    _pair(binding, golden, "lr_exclude", tmp_path)
