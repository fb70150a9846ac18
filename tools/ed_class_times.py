"""Per-class kernel times of the short-probe HW realign path at the K1 shape (bench.py's batch), so that a change can be attributed to a class.

For each word class c (probe rows 32(c-1)+1 .. 32c) two sub-batches are cut from one K1 batch:
  pair c    the (ALT, REF) job pairs whose longer probe is in class c, kept adjacent: they run as pairs (ed_hw_kernel<c, 2>)
  single c  the jobs of class c in an order where no two neighbours share a read: they run one per thread
Each is run through the device form with the async bound set (as bench.py does), and the library's own CUDA events around its kernels
(dgpu_set_profiling / dgpu_last_kernel_ms) give the time; the median over --reps runs is reported per job. DGPU_LIB selects another
build of the library (a library without pair classes runs the pair batches one job per thread).

usage: python tools/ed_class_times.py [--jobs 2000000] [--reps 20] [--out FILE.json]
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--jobs", type=int, default=2_000_000)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    import delly_b200
    from delly_b200 import synth

    b = synth.k1_genotype_batch(args.jobs, seed=1001)
    n = len(b["q_len"]) // 2 * 2
    qa, qb = b["q_len"][0:n:2].astype(np.int64), b["q_len"][1:n:2].astype(np.int64)
    pair_cls = (np.maximum(qa, qb) + 31) // 32
    job_cls = (b["q_len"][:n].astype(np.int64) + 31) // 32
    dev = torch.device("cuda", 0)
    ctx = delly_b200.Context(0)
    ctx.set_profiling(True)
    seqs = torch.from_numpy(b["seqs"]).to(dev)
    ctx.check(delly_b200.lib().dgpu_set_async_bound(ctx.h, 256), "dgpu_set_async_bound")
    stream = torch.cuda.current_stream().cuda_stream

    def run(idx):
        t = {k: torch.from_numpy(np.ascontiguousarray(b[k][idx])).to(dev) for k in ("q_off", "q_len", "t_off", "t_len", "k")}
        out = torch.empty(len(idx), dtype=torch.int32, device=dev)
        for _ in range(3):
            ctx.edit_distance_dev(seqs, t["q_off"], t["q_len"], t["t_off"], t["t_len"], t["k"], delly_b200.MODE_HW, out, None, stream)
        torch.cuda.synchronize()
        ms = []
        for _ in range(args.reps):
            ctx.edit_distance_dev(seqs, t["q_off"], t["q_len"], t["t_off"], t["t_len"], t["k"], delly_b200.MODE_HW, out, None, stream)
            ms.append(ctx.last_kernel_ms())
        return float(np.median(ms)), float(np.min(ms)), float(np.max(ms))

    rows = []
    for c in (1, 2, 3, 4):
        pj = np.nonzero(pair_cls == c)[0]
        if len(pj):
            idx = np.stack([2 * pj, 2 * pj + 1], axis=1).reshape(-1)
            med, lo, hi = run(idx)
            rows.append({"class": f"pair {c}", "jobs": int(len(idx)), "ms": med, "ms_min": lo, "ms_max": hi, "ns_per_job": med * 1e6 / len(idx)})
        sj = np.nonzero(job_cls == c)[0]
        if len(sj):
            idx = np.concatenate([sj[sj % 2 == 0], sj[sj % 2 == 1]])   # neighbours are different reads: no pairs
            med, lo, hi = run(idx)
            rows.append({"class": f"single {c}", "jobs": int(len(idx)), "ms": med, "ms_min": lo, "ms_max": hi, "ns_per_job": med * 1e6 / len(idx)})
    ctx.check(delly_b200.lib().dgpu_set_async_bound(ctx.h, 0), "dgpu_set_async_bound")
    res = {"lib": delly_b200.LIB_PATH, "gpu": torch.cuda.get_device_name(0), "jobs": args.jobs, "reps": args.reps, "classes": rows}
    for r in rows:
        print(f"{r['class']:>9}  {r['jobs']:>9} jobs  {r['ms']:8.3f} ms  [{r['ms_min']:.3f}, {r['ms_max']:.3f}]  {r['ns_per_job']:7.4f} ns/job")
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    ctx.close()


if __name__ == "__main__":
    main()
