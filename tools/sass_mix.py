"""Static instruction mix of the fast path of the short-probe HW realign kernels, per DP column per job, split by pipe.

Compiles delly_b200/csrc/edit_distance.cu (or --src FILE, e.g. an older version of it) for sm_100a, disassembles it with cuobjdump -sass
and, in each HW distance kernel (ed_hw_kernel<NW, J>, and ed_small_kernel<NW, HW, false> where a version still has it), finds the target
chunk loop: the smallest loop (backward branch) that holds at least 16*NW shared-memory loads, i.e. one 16-column chunk of Peq reads.
Inside it the counted blocks are
  - the four-column fast blocks (straight-line blocks with >= 4*NW LDS: four columns of Peq loads and Myers updates),
  - the block right before each of them (the four-byte ACGT check and the branch to the exact slow path),
  - the blocks that load and realign the next 16 target bytes (LDG.128) and the loop latch.
The slow path for bytes outside ACGT (and anything else the loop holds) is not counted. The total is divided by 16 columns and by J
jobs per thread. Pipes: FMA = IMAD* / FFMA / FMUL / FADD / HFMA2 (integer multiply-add forms run there), ALU = LOP3, IADD3, SHF, ISETP,
SEL, PRMT, LEA, IMNMX, MOV, ... ; other = memory and control. ptxas decides the final form, so this is read from the SASS, not the source.

usage: python tools/sass_mix.py [--src FILE] [--verbose]
"""
import argparse
import collections
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
CUOBJDUMP = os.path.join(os.path.dirname(NVCC), "cuobjdump")

FMA = ("IMAD", "FFMA", "FMUL", "FADD", "HFMA2", "HMUL2", "HADD2")
ALU = ("LOP3", "IADD3", "IADD", "SHF", "ISETP", "SEL", "PRMT", "LEA", "IMNMX", "VIMNMX", "VIADD", "MOV", "IABS", "POPC", "FLO", "BMSK",
       "SGXT", "PLOP3", "P2R", "R2P", "LOP", "FSEL", "ICMP", "BREV", "UIADD3", "UMOV", "ULOP3", "USHF", "ISCADD", "IADD32I", "LOP32I")
LINE = re.compile(r"/\*([0-9a-f]{4,})\*/\s+(.*?)\s*;")


def compile_sass(src):
    with tempfile.TemporaryDirectory() as d:
        cubin = os.path.join(d, "ed.cubin")
        subprocess.check_call([NVCC, "-std=c++17", "-O3", "-cubin", "-gencode", "arch=compute_100a,code=sm_100a",
                               "-I", os.path.join(ROOT, "delly_b200", "csrc"), "-I", os.path.join(ROOT, "include"), "-o", cubin, src])
        return subprocess.check_output([CUOBJDUMP, "-sass", cubin], text=True)


def functions(sass):
    cur, out = None, {}
    for line in sass.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            cur = m.group(1)
            out[cur] = []
            continue
        if cur is None:
            continue
        m = LINE.search(line)
        if m:
            addr = int(m.group(1), 16)
            text = m.group(2).strip()
            pred = ""
            if text.startswith("@"):
                pred, text = text.split(None, 1)
            op = text.split()[0]
            tgt = None
            if op.startswith("BRA"):
                t = re.search(r"0x([0-9a-f]+)", text)
                tgt = int(t.group(1), 16) if t else None
            out[cur].append((addr, op, pred, tgt))
    return out


def pipe(op):
    base = op.split(".")[0]
    if base.startswith(FMA):
        return "FMA"
    if base in ALU:
        return "ALU"
    return "other"


def chunk_loop_mix(ins, nw, j):
    lds = lambda o: o.startswith("LDS")
    loops = [(tgt, a) for a, op, _, tgt in ins if op.startswith("BRA") and tgt is not None and tgt < a]
    best = None
    for lo, hi in loops:
        body = [x for x in ins if lo <= x[0] <= hi]
        if sum(lds(x[1]) for x in body) >= 16 * nw and (best is None or hi - lo < best[1] - best[0]):
            best = (lo, hi)
    if best is None:
        return None
    lo, hi = best
    body = [x for x in ins if lo <= x[0] <= hi]
    leaders = {lo} | {x[3] for x in body if x[3] is not None and lo <= x[3] <= hi}
    blocks, cur = [], []
    for x in body:
        if x[0] in leaders and cur:
            blocks.append(cur)
            cur = []
        cur.append(x)
        if x[1].startswith(("BRA", "EXIT", "RET")):
            blocks.append(cur)
            cur = []
    if cur:
        blocks.append(cur)
    take = set()
    for i, b in enumerate(blocks):
        n_lds = sum(lds(x[1]) for x in b)
        if n_lds >= 4 * nw:
            take.add(i)
            if i > 0 and not any(lds(x[1]) for x in blocks[i - 1]):
                take.add(i - 1)
        if any(x[1].startswith("LDG") and ".128" in x[1] for x in b) or any(x[0] == hi for x in b):
            take.add(i)
    cnt = collections.Counter()
    for i in sorted(take):
        for x in blocks[i]:
            if not x[1].startswith("NOP"):
                cnt[x[1]] += 1
    per = 16.0 * j
    by_pipe = collections.Counter()
    for op, c in cnt.items():
        by_pipe[pipe(op)] += c
    return {"fast_blocks": sum(1 for i in take if sum(lds(x[1]) for x in blocks[i]) >= 4 * nw),
            "ops": {op: c / per for op, c in cnt.items()}, "pipes": {p: c / per for p, c in by_pipe.items()},
            "total": sum(cnt.values()) / per}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--src", default=os.path.join(ROOT, "delly_b200", "csrc", "edit_distance.cu"))
    ap.add_argument("--verbose", action="store_true")
    args = ap.parse_args()
    fns = functions(compile_sass(os.path.abspath(args.src)))
    rows = []
    for name, ins in fns.items():
        m = re.search(r"ed_hw_kernelILi(\d)ELi(\d)E", name)
        if m:
            label, nw, j = f"ed_hw_kernel<{m.group(1)},{m.group(2)}>", int(m.group(1)), int(m.group(2))
        else:
            m = re.search(r"ed_small_kernelILi(\d)ELi2ELb0E", name)
            if not m:
                continue
            label, nw, j = f"ed_small_kernel<{m.group(1)},HW,false>", int(m.group(1)), 1
        r = chunk_loop_mix(ins, nw, j)
        rows.append((label, nw, j, r))
    print(f"{'kernel':<26} {'inst/col/job':>12} {'ALU':>7} {'FMA':>7} {'other':>7}  fast blocks")
    for label, nw, j, r in sorted(rows, key=lambda x: (x[0].split("<")[0], x[1], x[2])):
        if r is None:
            print(f"{label:<26} no chunk loop found")
            continue
        p = r["pipes"]
        print(f"{label:<26} {r['total']:12.2f} {p.get('ALU', 0):7.2f} {p.get('FMA', 0):7.2f} {p.get('other', 0):7.2f}  {r['fast_blocks']}")
        if args.verbose:
            for op, c in sorted(r["ops"].items(), key=lambda kv: -kv[1]):
                print(f"    {op:<22} {pipe(op):<5} {c:6.2f}")
    return 0


if __name__ == "__main__":
    sys.exit(main())
