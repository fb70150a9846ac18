#!/usr/bin/env python
"""Build step: writes the template sequences of the reference's long-read annotation (class MEI, src/svanno.h:30-39 — consensus
sequences of Alu, LINE-1, SVA, the mitochondrial genome, a solo LTR, HERV-K and a poly-A tail; data, not code) into a FASTA next to the
reference's other build products (oracle/_ref/mei_templates.fa) and puts a copy next to the product binary (delly_b200/data/_mei_templates.fa).
Both are git-ignored. Where the reference tree is absent, the copy is made from an oracle/_ref built elsewhere. `delly_b200 lr` reads it (or
the file given with --mei)."""
import os
import re
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get("REF", "/root/reference")
src = os.path.join(REF, "src", "svanno.h")
staged = os.path.join(ROOT, "oracle", "_ref", "mei_templates.fa")
out = os.path.join(ROOT, "delly_b200", "data", "_mei_templates.fa")


def install():
    os.makedirs(os.path.dirname(out), exist_ok=True)
    with open(staged) as f, open(out, "w") as g:
        g.write(f.read())


if not os.path.exists(src):
    if os.path.exists(staged):
        install()
        print("reference not present; copied", staged, "to", out)
    else:
        print("reference not present and", staged, "missing; keeping", out)
    sys.exit(0)
text = open(src).read()
body = text[text.index("class MEI"):]
body = body[:body.index("};")]
recs = re.findall(r'std::string\s+(\w+)\s*=\s*((?:"[A-Za-z]*"\s*)+);', body)
assert len(recs) == 7, [r[0] for r in recs]
os.makedirs(os.path.dirname(staged), exist_ok=True)
with open(staged, "w") as f:
    for name, lit in recs:
        seq = "".join(re.findall(r'"([A-Za-z]*)"', lit))
        f.write(">%s\n%s\n" % (name, seq))
install()
print("wrote", staged, "and", out, {n: len("".join(re.findall(r'"([A-Za-z]*)"', l))) for n, l in recs})
