"""Writes tests/golden/bcf_parity.npz: what the reference's own drivers (oracle/_ref/delly_ref) write for every case of
tests/test_bcf_parity.py on the reference's example data (oracle/_ref/example). Both need a build where the reference tree exists.

    python tests/golden/make_bcf_parity.py

Per case <c>: "<c>.bcf" the inflated BCF with the ##fileDate value replaced by X, "<c>.bcf.csi" its index. "sr.vcf" is the VCF text of
`delly sr -g ref.fa sr.bam` on stdout. "sr.sites.bcf" / "lr.sites.bcf" (+ ".csi") are the discovery outputs as written (BGZF): the site
lists the genotyping cases read back. Every array is the bytes as uint8."""
import os
import subprocess
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
import test_bcf_parity as t  # noqa: E402

DELLY_REF = os.path.join(t.REFDIR, "delly_ref")


def run(args):
    r = subprocess.run([DELLY_REF] + args, cwd=t.EX, capture_output=True)
    assert r.returncode == 0, (args, r.stderr[-2000:])
    return r.stdout


def main():
    out = {}
    with tempfile.TemporaryDirectory() as tmp:
        def sites(name):
            p = os.path.join(tmp, name + ".sites.bcf")
            if not os.path.exists(p):
                run(t.case_command(name, p, tmp, None))
                for ext in ("", ".csi"):
                    out[name + ".sites.bcf" + ext] = open(p + ext, "rb").read()
            return p

        for case in t.CASES:
            p = os.path.join(tmp, case + ".bcf")
            run(t.case_command(case, p, tmp, sites))
            out[case + ".bcf"] = t._inflate(p)
            out[case + ".bcf.csi"] = open(p + ".csi", "rb").read()
        out[t.VCF_TEXT_CASE + ".vcf"] = run(["sr", "-g", "ref.fa", "sr.bam"])
        for k, v in out.items():
            assert tmp.encode() not in v, k       # no path of this run inside the stored outputs
    np.savez_compressed(os.path.join(HERE, "bcf_parity.npz"), **{k: np.frombuffer(v, np.uint8) for k, v in out.items()})
    print({k: len(v) for k, v in out.items()})


if __name__ == "__main__":
    main()
