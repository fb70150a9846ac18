#!/usr/bin/env python
"""bench.py — split-read realigns/sec on the sr genotyping workload (BASELINE.json configs[1]).

One "step" = one pass of the hot path over one batch: every read overlapping a breakpoint is
realigned against its SV's ALT and REF probes (two infix edit-distance jobs per read,
src/coverage.h:412-441). configs[1] names ~5 M split/discordant reads -> 10 M realigns per step.

  value   realigns/s, inputs already resident in HBM (dgpu_edit_distance_dev on torch's stream)
  e2e     the same metric through the host-pointer C ABI call (pinned host buffers, H2D + D2H in the
          timed region)
  roofline      the dominant kernel family (ed_small_kernel<NW>) timed with CUDA events inside the
                library on the launching stream; HBM figure as the contract asks, plus the
                integer-pipe figure this path is actually bound by (roofline.bound = int32 ALU, HBM as roofline.hbm)
  cpu_baseline  the reference's own edlib (oracle/_ref, compiled verbatim) on all host cores, on a
                bounded sample of the same batch

Launch: python bench.py [--gpus N --steps K --warmup W] ; N>1 under torchrun (one rank per GPU).
        python bench.py --impl reference ...   times the reference CPU path on the same config.
        python bench.py --dump-outputs DIR ...  also writes what the last timed step computed to DIR (see dump_outputs;
                                                bench_outputs/ is git-ignored for this).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

JOBS_PER_STEP = 10_000_000
CHUNK = 100_000
METRIC = "split-read realigns/sec (sr genotyping: HW edit-distance realign of REF/ALT probe vs read)"
UNIT = "realigns/s"


def make_batch(n_jobs, seed):
    """configs[1]-shaped batch, generated in 1 M-job chunks (bounded host memory), one packed arena."""
    from delly_b200 import synth
    parts = []
    base = 0
    for c in range(0, n_jobs, CHUNK):
        b = synth.k1_genotype_batch(min(CHUNK, n_jobs - c), seed=seed + c // CHUNK, genome_len=500_000)
        b["q_off"] = (b["q_off"].astype(np.int64) + base).astype(np.uint32)
        b["t_off"] = (b["t_off"].astype(np.int64) + base).astype(np.uint32)
        base += len(b["seqs"])
        parts.append(b)
    assert base < 2 ** 32
    return {k: np.concatenate([p[k] for p in parts]) for k in parts[0]}


DUMP_BUDGET = 64 << 20
DUMP_SEED = 20240917


def dump_outputs(out_dir, dist, world, rank):
    """Writes the edit distances of the last timed step (what a caller of dgpu_edit_distance_dev receives, one int32 per job, -1 where the
    bound k was exceeded) as float32 to out_dir/edit_distance.npy (N > 1: edit_distance_rank<r>.npy per rank). The inputs are seeded, so two
    builds given the same arguments can be compared output for output. Above the 64 MB budget (shared by all ranks) a fixed, seeded sample
    of job indices is written instead, in job order, with the indices in edit_distance_index.npy (float64, exact)."""
    os.makedirs(out_dir, exist_ok=True)
    sfx = "" if world == 1 else f"_rank{rank}"
    n = len(dist)
    cap = DUMP_BUDGET // world // 4
    if n > cap:
        # indices (8 bytes each as float64) and values (4 bytes) share the budget
        idx = np.sort(np.random.default_rng(DUMP_SEED).choice(n, size=DUMP_BUDGET // world // 12, replace=False))
        np.save(os.path.join(out_dir, f"edit_distance_index{sfx}.npy"), idx.astype(np.float64))
        dist = dist[idx]
    np.save(os.path.join(out_dir, f"edit_distance{sfx}.npy"), dist.astype(np.float32))


def algorithmic_counts(b):
    """SURVEY.md §8(d): Myers = ceil(m/64)*n block-steps x 34 int32 ops; bytes = m + n in, 4 out per job
    (+ the 20 B of job metadata the kernel must read: 2 offsets, 2 lengths, k)."""
    m = b["q_len"].astype(np.int64)
    n = b["t_len"].astype(np.int64)
    ops = int((((m + 63) // 64) * n * 34).sum())
    byts = int((m + n + 4 + 20).sum())
    cells = int((m * n).sum())
    return ops, byts, cells


class ClockSampler:
    """SM clock + throttle reasons sampled DURING the timed region (NVML, ~2 ms period; nvidia-smi fallback)."""

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.sm, self.reasons, self.mx = [], set(), None
        self._stop = threading.Event()
        self.t = None
        self.err = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[self.idx]) if vis and vis.split(",")[self.idx].isdigit() else self.idx
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.mx = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.t = threading.Thread(target=self._loop, daemon=True)
            self.t.start()
        except Exception as e:  # noqa: BLE001
            self.err = repr(e)

    def _loop(self):
        nv = self.nv
        names = {"hw_slowdown": nv.nvmlClocksThrottleReasonHwSlowdown,
                 "hw_thermal_slowdown": nv.nvmlClocksThrottleReasonHwThermalSlowdown,
                 "sw_thermal_slowdown": nv.nvmlClocksThrottleReasonSwThermalSlowdown,
                 "sw_power_cap": nv.nvmlClocksThrottleReasonSwPowerCap}
        while not self._stop.is_set():
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception as e:  # noqa: BLE001
                self.err = repr(e)
                break
            time.sleep(0.002)

    def stop(self):
        self._stop.set()
        if self.t:
            self.t.join(timeout=2)
        out = {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.mx,
               "reasons": sorted(self.reasons), "samples": len(self.sm)}
        if self.err:
            out["sampler_error"] = self.err
        return out


def host_cores():
    """threads this process may actually use (cgroup / affinity aware; os.cpu_count() is not)"""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return os.cpu_count() or 1


def cpu_reference_leg(b, target_seconds=6.0, full=False, repeats=3):
    """Time the reference's edlib (oracle/_ref) — or the oracle port if _ref is absent — on the host cores: the reference's worker
    scheme (fixed pool pulling an atomic index, src/coverage.h:412-441). full=False: a bounded sample (about target_seconds of work);
    full=True: the whole step batch. Best of `repeats` runs (the pool's rate swings with what else the box is doing); per-core rate too."""
    from oracle import pyoracle as po
    lib = po.ref()
    kind = "reference" if lib is not None else "port"
    if lib is None:
        lib = po.oracle()
    cores = host_cores()
    n = len(b["q_off"])

    def run(cnt):
        sub = {k: (v if k == "seqs" else v[:cnt]) for k, v in b.items()}
        t0 = time.perf_counter()
        d, _ = po.edit_distance_batch(lib, sub["seqs"], sub["q_off"], sub["q_len"], sub["t_off"], sub["t_len"], sub["k"], 2,
                                      threads=cores)
        return time.perf_counter() - t0, d

    if full:
        cnt = n
    else:
        pilot = min(n, 20000 * cores)
        t, _ = run(pilot)
        rate = pilot / max(t, 1e-6)
        cnt = int(min(n, max(pilot, rate * target_seconds / repeats)))
    times, d = [], None
    for _ in range(repeats):
        t, d = run(cnt)
        times.append(t)
    t = min(times)
    return {"value": cnt / t, "unit": UNIT, "cores": cores, "kind": kind, "per_core": cnt / t / cores, "runs_s": [round(x, 4) for x in times],
            "sample": f"{'all' if cnt == n else 'first'} {cnt} of {n} jobs of the step batch, best of {repeats} runs ({t:.2f} s wall) on {cores} threads "
                      f"(atomic-index worker pool as src/coverage.h:412-441)"}, d, cnt, t


def bench_families(ctx, reps=3):
    """Kernel-family throughputs beside the headline (never mixed into it): K3 = sr longNeedle
    (cons 150-300 vs SV window 600-1600), K2 = sr msa clusters (2-20 reads x 150 bp). Device time = library-side
    CUDA events around the family's kernels; e2e = host-pointer ABI call; cpu = compiled reference on all cores."""
    import ctypes as C
    from delly_b200 import synth, _ptr as delly_b200_ptr
    from oracle import pyoracle as po
    R = po.ref()
    cores = host_cores()
    out = []
    # ---- K3: longNeedle -------------------------------------------------------------------
    b = synth.k3_consref_batch(4096, seed=1003, cons_range=(150, 300), err=0.01, fast=True)
    rep = 12  # 49,152 jobs per call: the 4096 unique jobs replicated (inputs are tiny next to the DP work)
    c_off, c_len = np.tile(b["c_off"], rep), np.tile(b["c_len"], rep)
    r_off, r_len = np.tile(b["r_off"], rep), np.tile(b["r_len"], rep)
    n = len(c_off)
    cells = int(((c_len.astype(np.int64) + 1) * (r_len.astype(np.int64) + 1)).sum())
    ts, ks = [], []
    for i in range(reps + 1):
        t0 = time.perf_counter()
        ok, alen, _rows = ctx.long_needle(b["seqs"], c_off, c_len, r_off, r_len) if i == 0 else (None, None, None)
        if i > 0:
            cap = (c_len.astype(np.uint64) + r_len.astype(np.uint64))
            aln_off = np.concatenate([[0], np.cumsum(2 * cap)[:-1]]).astype(np.uint64)
            aln = np.empty(int(2 * cap.sum()), np.uint8); al = np.empty(n, np.uint32); okk = np.empty(n, np.uint8)
            t0 = time.perf_counter()
            rc = ctx._lib.dgpu_long_needle(ctx.h, C.c_void_p(b["seqs"].ctypes.data), C.c_uint64(b["seqs"].nbytes),
                                           C.c_void_p(c_off.ctypes.data), C.c_void_p(c_len.ctypes.data), C.c_void_p(r_off.ctypes.data),
                                           C.c_void_p(r_len.ctypes.data), C.c_uint64(n), C.c_void_p(aln.ctypes.data),
                                           C.c_void_p(aln_off.ctypes.data), C.c_uint64(aln.nbytes), C.c_void_p(al.ctypes.data),
                                           C.c_void_p(okk.ctypes.data), C.c_void_p(0))
            ctx.check(rc, "dgpu_long_needle")
            ts.append(time.perf_counter() - t0); ks.append(ctx.last_kernel_ms())
    kms = float(np.median(ks)); e2e = float(np.median(ts))
    fam = {"family": "K3 longNeedle (sr): consensus 150-300 bp vs SV window 600-1600 bp", "jobs": n, "unit": "alignments/s",
           "value": n / (kms * 1e-3), "kernel_ms": kms, "e2e_value": n / e2e,
           "gcups": 3 * cells / (kms * 1e-3) / 1e9, "int_ops_per_cell_algorithmic": 14,
           "achieved_tera_int_ops": 14 * cells / (kms * 1e-3) / 1e12}
    if R is not None:
        cnt = min(n, 64 * cores)
        okr = np.zeros(cnt, np.uint8); alr = np.zeros(cnt, np.uint32)
        co64, ro64 = c_off[:cnt].astype(np.uint64), r_off[:cnt].astype(np.uint64)  # keep alive across the call
        cl32, rl32 = np.ascontiguousarray(c_len[:cnt]), np.ascontiguousarray(r_len[:cnt])
        t0 = time.perf_counter()
        R.ref_long_needle_batch(C.c_char_p(b["seqs"].ctypes.data), C.c_void_p(co64.ctypes.data),
                                C.c_void_p(cl32.ctypes.data), C.c_void_p(ro64.ctypes.data),
                                C.c_void_p(rl32.ctypes.data), C.c_uint64(cnt), C.c_void_p(okr.ctypes.data),
                                C.c_void_p(alr.ctypes.data), cores)
        dt = time.perf_counter() - t0
        assert np.array_equal(okr, okk[:cnt]) and np.array_equal(alr, al[:cnt]), "K3: GPU differs from reference"
        fam["cpu_baseline"] = {"value": cnt / dt, "unit": "alignments/s", "cores": cores, "kind": "reference", "sample": f"{cnt} jobs, {dt:.2f} s"}
    out.append(fam)
    # ---- K2: msa ---------------------------------------------------------------------------------
    b = synth.k2_msa_batch(2048, seed=1002, fast=True)
    ncl = len(b["cluster_off"]) - 1
    rep = 24  # 49,152 clusters per call (SURVEY section 8d: K2 = 50 k): the 2048 unique clusters replicated
    nreads = len(b["read_off"])
    read_off = np.tile(b["read_off"], rep); read_len = np.tile(b["read_len"], rep)
    coff = np.concatenate([b["cluster_off"][:-1].astype(np.int64) + r * nreads for r in range(rep)] + [[rep * nreads]]).astype(np.uint32)
    N = len(coff) - 1
    ts, ks = [], []
    cons = None
    for i in range(reps + 1):
        t0 = time.perf_counter()
        cons, nrows, status = ctx.msa(b["seqs"], read_off, read_len, coff)
        ts.append(time.perf_counter() - t0); ks.append(ctx.last_kernel_ms())
    kms = float(np.median(ks[1:])); e2e = float(np.median(ts[1:]))
    fam = {"family": "K2 msa (sr): 2-20 reads x 150 bp per cluster (LCS + UPGMA + progressive gotoh + consensus)",
           "jobs": N, "unit": "clusters/s", "value": N / (kms * 1e-3), "kernel_ms": kms, "e2e_value": N / e2e}
    if R is not None:
        cnt = min(N, 8 * cores)
        rl = read_len.astype(np.uint64); csum = np.concatenate([[0], np.cumsum(rl)])
        cap = csum[coff[1:cnt + 1]] - csum[coff[:cnt]]
        cons_off = np.concatenate([[0], np.cumsum(cap)[:-1]]).astype(np.uint64)
        cbuf = np.zeros(int(cap.sum()), np.uint8); clen = np.zeros(cnt, np.uint32)
        ro64 = read_off.astype(np.uint64)  # keep alive across the call
        t0 = time.perf_counter()
        R.ref_msa_batch(C.c_char_p(b["seqs"].ctypes.data), C.c_void_p(ro64.ctypes.data), C.c_void_p(read_len.ctypes.data),
                        C.c_void_p(coff.ctypes.data), C.c_uint32(cnt), 2, 5, -4, -10, -1, C.c_char_p(cbuf.ctypes.data),
                        C.c_void_p(cons_off.ctypes.data), C.c_void_p(clen.ctypes.data), cores)
        dt = time.perf_counter() - t0
        for i in range(cnt):
            assert cons[i] == cbuf[int(cons_off[i]):int(cons_off[i]) + int(clen[i])].tobytes(), "K2: GPU consensus differs from reference"
        fam["cpu_baseline"] = {"value": cnt / dt, "unit": "clusters/s", "cores": cores, "kind": "reference", "sample": f"{cnt} clusters, {dt:.2f} s"}
    out.append(fam)
    # ---- K5: long-read longNeedle (consensus 2-4 kb vs SV window 4-16 kb) and K6: long-read NW edit distance -------------------
    b = synth.k3_consref_batch(1184, seed=2001, cons_range=(2000, 4000), err=0.05, fast=True, genome_len=4_000_000)  # 8 CTA waves (one 8-warp CTA per SM)
    rep5 = 21   # 24,864 jobs per call (SURVEY section 8d: K5 = 25 k): the 1184 unique jobs replicated; device form, results stay on the device
    import torch
    dv = torch.device("cuda", ctx.device)
    c_off5, c_len5 = np.tile(b["c_off"], rep5), np.tile(b["c_len"], rep5)
    r_off5, r_len5 = np.tile(b["r_off"], rep5), np.tile(b["r_len"], rep5)
    cells = int(((c_len5.astype(np.int64) + 1) * (r_len5.astype(np.int64) + 1)).sum())
    cap5 = c_len5.astype(np.uint64) + r_len5.astype(np.uint64)
    aoff5 = np.concatenate([[0], np.cumsum(2 * cap5)[:-1]]).astype(np.int64)
    tt = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dv)
    d5 = dict(seqs=tt(np.concatenate([b["seqs"], np.zeros(64, np.uint8)])), c_off=tt(c_off5.view(np.int32)), c_len=tt(c_len5.view(np.int32)), r_off=tt(r_off5.view(np.int32)),
              r_len=tt(r_len5.view(np.int32)), aoff=tt(aoff5), aln=torch.empty(int(2 * cap5.sum()) + 64, dtype=torch.uint8, device=dv),
              alen=torch.empty(len(c_off5), dtype=torch.int32, device=dv), ok=torch.empty(len(c_off5), dtype=torch.uint8, device=dv))
    ks = []
    for i in range(2):
        rc = ctx._lib.dgpu_long_needle_dev(ctx.h, delly_b200_ptr(d5["seqs"]), C.c_uint64(len(b["seqs"])), delly_b200_ptr(d5["c_off"]), delly_b200_ptr(d5["c_len"]),
                                           delly_b200_ptr(d5["r_off"]), delly_b200_ptr(d5["r_len"]), C.c_uint64(len(c_off5)), delly_b200_ptr(d5["aln"]),
                                           delly_b200_ptr(d5["aoff"]), delly_b200_ptr(d5["alen"]), delly_b200_ptr(d5["ok"]), C.c_void_p(0), C.c_void_p(0))
        ctx.check(rc, "dgpu_long_needle_dev"); torch.cuda.synchronize(); ks.append(ctx.last_kernel_ms())
    kms = float(min(ks))
    okk, al = d5["ok"].cpu().numpy()[:len(b["c_off"])], d5["alen"].cpu().numpy().view(np.uint32)[:len(b["c_off"])]
    n5 = len(c_off5)
    del d5
    fam = {"family": "K5 longNeedle (lr): consensus 2-4 kb vs SV window 4-16 kb", "jobs": n5, "unit": "alignments/s",
           "value": n5 / (kms * 1e-3), "kernel_ms": kms, "gcups": 3 * cells / (kms * 1e-3) / 1e9, "int_ops_per_cell_algorithmic": 14,
           "achieved_tera_int_ops": 14 * cells / (kms * 1e-3) / 1e12}
    if R is not None:
        cnt = min(len(okk), max(4, cores // 8))
        okr = np.zeros(cnt, np.uint8); alr = np.zeros(cnt, np.uint32)
        co64, ro64 = b["c_off"][:cnt].astype(np.uint64), b["r_off"][:cnt].astype(np.uint64)
        cl32, rl32 = np.ascontiguousarray(b["c_len"][:cnt]), np.ascontiguousarray(b["r_len"][:cnt])
        t0 = time.perf_counter()
        R.ref_long_needle_batch(C.c_char_p(b["seqs"].ctypes.data), C.c_void_p(co64.ctypes.data), C.c_void_p(cl32.ctypes.data), C.c_void_p(ro64.ctypes.data),
                                C.c_void_p(rl32.ctypes.data), C.c_uint64(cnt), C.c_void_p(okr.ctypes.data), C.c_void_p(alr.ctypes.data), cnt)
        dt = time.perf_counter() - t0
        assert np.array_equal(okr, okk[:cnt]) and np.array_equal(alr, al[:cnt]), "K5: GPU differs from reference"
        fam["cpu_baseline"] = {"value": cnt / dt, "unit": "alignments/s", "cores": cnt, "kind": "reference", "sample": f"{cnt} jobs on {cnt} threads, {dt:.2f} s (delly lr itself is single-threaded)"}
    out.append(fam)
    rng = np.random.default_rng(2002)
    seqs = []
    for _ in range(20000):
        L = int(rng.integers(200, 4001)); t = synth._ACGT[rng.integers(0, 4, size=L, dtype=np.uint8)]
        seqs += [synth.sub_noise(rng, t, 0.08), t]
    arena, off, ln = synth.pack(seqs)
    q_off, q_len, t_off, t_len = off[0::2].copy(), ln[0::2].copy(), off[1::2].copy(), ln[1::2].copy()
    rep6 = 100   # 2 M jobs per call (SURVEY section 8d: K6 = 2 M): the 20,000 unique pairs replicated (offsets into the same arena)
    q_off, q_len, t_off, t_len = np.tile(q_off, rep6), np.tile(q_len, rep6), np.tile(t_off, rep6), np.tile(t_len, rep6)
    kk = np.full(len(q_off), -1, np.int32)
    # device form, timed with CUDA events on the launching stream (the host form uploads in pieces and its kernel span covers the last piece only)
    t6 = {k: tt(v) for k, v in (("seqs", np.concatenate([arena, np.zeros(64, np.uint8)])), ("q_off", q_off.view(np.int32)), ("q_len", q_len.view(np.int32)),
                                ("t_off", t_off.view(np.int32)), ("t_len", t_len.view(np.int32)), ("k", kk))}
    d6 = torch.empty(len(q_off), dtype=torch.int32, device=dv)
    ks = []
    for i in range(3):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        ctx.edit_distance_dev(t6["seqs"][:len(arena)], t6["q_off"], t6["q_len"], t6["t_off"], t6["t_len"], t6["k"], 0, d6, None, torch.cuda.current_stream().cuda_stream)
        e1.record(); torch.cuda.synchronize()
        ks.append(e0.elapsed_time(e1))
    kms = float(min(ks))
    dd = d6.cpu().numpy()
    del t6, d6
    cells = int((q_len.astype(np.int64) * t_len.astype(np.int64)).sum())
    fam = {"family": "K6 edit distance NW (lr): 200-4000 bp vs same, 8 % substitutions", "jobs": len(dd), "unit": "alignments/s",
           "value": len(dd) / (kms * 1e-3), "kernel_ms": kms, "gcups": cells / (kms * 1e-3) / 1e9}
    if R is not None:
        cnt = min(len(dd), 200 * cores)
        t0 = time.perf_counter()
        rd, _ = po.edit_distance_batch(R, arena, q_off[:cnt], q_len[:cnt], t_off[:cnt], t_len[:cnt], kk[:cnt], 0, threads=cores)
        dt = time.perf_counter() - t0
        assert np.array_equal(rd, dd[:cnt]), "K6: GPU differs from reference"
        fam["cpu_baseline"] = {"value": cnt / dt, "unit": "alignments/s", "cores": cores, "kind": "reference", "sample": f"{cnt} jobs, {dt:.2f} s"}
    out.append(fam)
    # ---- K8: split-read clustering (src/cluster.h:324-442): pair scan on the device + sequential clique search on the host ----
    try:
        import delly_b200
        H = delly_b200.hostlib(); R2 = po.ref2()
        rng = np.random.default_rng(3003)
        ncl = 150_000  # planted deletion junctions, 1-11 supporting split reads each, plus unrelated records
        k = rng.integers(1, 12, size=ncl); tot = int(k.sum())
        base = np.repeat(rng.integers(1000, 60_000_000, size=ncl), k); size = np.repeat(rng.integers(20, 5000, size=ncl), k)
        chrs = np.repeat(rng.integers(0, 3, size=ncl), k)
        rows = np.zeros((tot + 200_000, 8), np.int32)
        rows[:tot, 0] = chrs; rows[:tot, 1] = base + rng.integers(-10, 11, size=tot); rows[:tot, 2] = chrs
        rows[:tot, 3] = base + size + rng.integers(-10, 11, size=tot)
        nz = len(rows) - tot
        rows[tot:, 0] = rng.integers(0, 3, size=nz); rows[tot:, 1] = rng.integers(1000, 60_000_000, size=nz); rows[tot:, 2] = rows[tot:, 0]
        rows[tot:, 3] = rows[tot:, 1] + rng.integers(1, 8000, size=nz)
        rows[:, 4] = rng.integers(0, 1000, size=len(rows)); rows[:, 5] = rng.integers(0, 150, size=len(rows)); rows[:, 6] = rng.integers(0, 61, size=len(rows))
        ids = (np.arange(len(rows), dtype=np.uint64) * 5 + 10)
        order = np.lexsort((rows[:, 3], rows[:, 2], rows[:, 1], rows[:, 0]))
        rows = np.ascontiguousarray(rows[order]); ids = np.ascontiguousarray(ids[order])
        n = len(rows); cap = 400_000
        svid = np.zeros(n, np.int32); sv = np.zeros((cap, 14), np.int32)
        ts, ks = [], []
        for i in range(3):
            t0 = time.perf_counter()
            cnt = H.dh_cluster_sr_gpu(ctx.h, C.c_void_p(rows.ctypes.data), C.c_void_p(ids.ctypes.data), n, 2, 2, 40, 1000, 3, C.c_void_p(svid.ctypes.data),
                                      C.c_void_p(sv.ctypes.data), cap)
            ts.append(time.perf_counter() - t0); ks.append(ctx.last_kernel_ms())
        assert cnt > 0, cnt
        fam = {"family": "K8 SR clustering (cluster(), svt 2): pair scan on the device (count/scan/fill), component + clique search on the host",
               "jobs": n, "unit": "records/s", "value": n / float(np.median(ts)), "kernel_ms": float(np.median(ks)),
               "edge_kernel_records_per_s": n / (float(np.median(ks)) * 1e-3), "svs": int(cnt)}
        if R2 is not None:
            svid2 = np.zeros(n, np.int32); sv2 = np.zeros((cap, 14), np.int32)
            t0 = time.perf_counter()
            cnt2 = R2.ref_cluster_sr(C.c_void_p(rows.ctypes.data), C.c_void_p(ids.ctypes.data), n, 2, 2, 40, 1000, 3, C.c_void_p(svid2.ctypes.data),
                                     C.c_void_p(sv2.ctypes.data), cap)
            dt = time.perf_counter() - t0
            assert cnt2 == cnt and np.array_equal(svid, svid2) and np.array_equal(sv[:cnt], sv2[:cnt]), "K8: GPU clustering differs from reference"
            fam["cpu_baseline"] = {"value": n / dt, "unit": "records/s", "cores": 1, "kind": "reference", "sample": f"{n} records, {dt:.2f} s (cluster() is serial in the reference)"}
        out.append(fam)
    except Exception as e:  # the family is auxiliary: report, never break the headline line
        out.append({"family": "K8 SR clustering", "error": repr(e)})
    # ---- K4: insertion consensus alignment (splitAlign, src/split.h:480-537: six edlib PATH calls per case + the glue), SURVEY section 8d: 5 k cases ----
    try:
        import delly_b200
        H = delly_b200.hostlib(); Rr = po.ref()
        rng = np.random.default_rng(1004)
        g = synth._ACGT[rng.integers(0, 4, size=2_000_000)]
        seqs = []
        n4 = 5000
        for it in range(n4):
            L = int(rng.integers(60, 140)); ins = int(rng.integers(20, 150)); p = int(rng.integers(10000, len(g) - 10000))
            cons = np.concatenate([g[p - L:p], synth._ACGT[rng.integers(0, 4, size=ins)], g[p:p + L]])
            if it % 3 == 0:
                cons = synth.mutate_fast(rng, cons, sub=0.01, ins=0.004, dele=0.004)
            w = max((len(cons) - ins) // 3, 13)
            seqs += [cons, g[p - w:p + 1 + w]]
        arena, off, ln = synth.pack(seqs)
        co, cl, ro, rl = off[0::2].copy(), ln[0::2].copy(), off[1::2].copy(), ln[1::2].copy()
        okv = np.zeros(n4, np.uint8); alv = np.zeros(n4, np.int32)
        P = lambda a: C.c_void_p(a.ctypes.data)
        ts = []
        for i in range(3):
            t0 = time.perf_counter()
            rc = H.dh_split_align_batch(ctx.h, P(arena), P(co), P(cl), P(ro), P(rl), n4, P(okv), P(alv))
            ts.append(time.perf_counter() - t0)
            assert rc == 0, rc
        fam = {"family": "K4 splitAlign (sr insertions): consensus 140-430 bp vs two-sided reference window, six edlib PATH calls + glue per case", "jobs": n4,
               "unit": "alignments/s", "value": n4 / float(np.median(ts)), "timing": "wall clock of the batched host call", "aligned": int(okv.sum())}
        if Rr is not None:
            chk = 300
            t0 = time.perf_counter()
            for i in range(chk):
                cb = arena[int(co[i]):int(co[i]) + int(cl[i])].tobytes(); rb = arena[int(ro[i]):int(ro[i]) + int(rl[i])].tobytes()
                rows = C.create_string_buffer(4 * (len(cb) + len(rb)) + 64); al = C.c_int()
                okk = Rr.ref_cons_ref_alignment(cb, len(cb), rb, len(rb), 4, rows, C.c_long(len(rows)), C.byref(al))
                assert (okk > 0) == bool(okv[i]) and (not okk or al.value == alv[i]), "K4: GPU differs from reference"
            dt = time.perf_counter() - t0
            fam["cpu_baseline"] = {"value": chk / dt, "unit": "alignments/s", "cores": 1, "kind": "reference", "sample": f"{chk} cases, {dt:.2f} s on one core (the reference spreads SVs over its -h worker threads)"}
        out.append(fam)
    except Exception as e:
        out.append({"family": "K4 splitAlign", "error": repr(e)})
    # ---- K7: long-read consensus (msaEdlib, src/assemble.h:385-473): all-pairs NW distances + progressive IUPAC-aware NW paths per cluster,
    #      batched over the clusters (host/msaedlib.hpp). Wall time of the host call (device rounds + host folding).
    try:
        import delly_b200
        H = delly_b200.hostlib(); R2 = po.ref2()
        rng = np.random.default_rng(2003)
        ncl = 960   # of section 8d's 25,000: enough to fill the device in every progressive round, and a call stays below a second
        reads, coff = [], [0]
        for _ in range(ncl):
            L = int(rng.integers(2000, 4000)); base = synth._ACGT[rng.integers(0, 4, size=L + 200)]
            for _ in range(15):
                a = int(rng.integers(0, 100)); r = base[a:a + L + int(rng.integers(-40, 40))]
                reads.append(synth.mutate_fast(rng, r, sub=0.03, ins=0.02, dele=0.02))
            coff.append(len(reads))
        arena, off, ln = synth.pack(reads)
        coff = np.array(coff, np.uint32)
        cons = np.zeros((ncl, 8192), np.uint8); clen = np.zeros(ncl, np.int32); rows = np.zeros(ncl, np.int32)
        P = lambda a: C.c_void_p(a.ctypes.data)
        ts = []
        for i in range(3):
            t0 = time.perf_counter()
            rc = H.dh_msa_edlib_batch(ctx.h, P(arena), P(off), P(ln), P(coff), ncl, 2, P(cons), 8192, P(clen), P(rows))
            ts.append(time.perf_counter() - t0)
            assert rc == 0, rc
        fam = {"family": "K7 msaEdlib (lr): 15 reads x 2-4 kb per cluster, 3 % sub + 4 % indel (all-pairs NW distance, progressive IUPAC-aware NW paths)",
               "jobs": ncl, "unit": "clusters/s", "value": ncl / float(np.median(ts)), "timing": "wall clock of the batched host call"}
        if R2 is not None:
            chk = 3
            t0 = time.perf_counter()
            for i in range(chk):
                a, b = int(coff[i]), int(coff[i + 1])
                buf = C.create_string_buffer(8192); cl = C.c_int()
                o2 = (off[a:b] - off[a]).astype(np.uint32); l2 = np.ascontiguousarray(ln[a:b])
                sub = np.ascontiguousarray(arena[int(off[a]):int(off[b - 1]) + int(ln[b - 1])])
                er = R2.ref_msa_edlib(P(sub), P(o2), P(l2), b - a, 2, buf, 8192, C.byref(cl))
                assert er == rows[i] and cons[i, :clen[i]].tobytes() == buf.raw[:cl.value], "K7: GPU consensus differs from reference"
            dt = time.perf_counter() - t0
            fam["cpu_baseline"] = {"value": chk / dt, "unit": "clusters/s", "cores": 1, "kind": "reference", "sample": f"{chk} clusters, {dt:.2f} s (msaEdlib is serial per SV in the reference)"}
        out.append(fam)
    except Exception as e:
        out.append({"family": "K7 msaEdlib", "error": repr(e)})
    return out


def workload_config(n, h2d_mb=None, world=1):
    """the `config` object of both arms (identical keys and values for the same --jobs)"""
    return {"workload": "configs[1]: sr genotyping realign, 5 M reads x (ALT,REF) probes = 10 M HW edit-distance jobs per step per GPU",
            "jobs_per_step_per_gpu": n, "probe_len": "U[26,80]", "read_len": 150, "k": "int(2*0.95f*|q|)",
            "l2": "inputs (959 MB/step at 10 M jobs) exceed the 126 MB L2; no flush needed",
            "parallelism": f"dp{world} (reads sharded by rank; per step one all-gatherv of the rank's call records)"}


def run_reference_arm(args):
    """The reference's own CPU implementation of the path (edlibAlign HW/DISTANCE through its worker-pool scheme, compiled verbatim from
    /root/reference into oracle/_ref) on all host threads, on the SAME step batch as the main arm: every step is the full batch, ms_per_step is
    measured."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    b = make_batch(args.jobs, seed=1001)
    n = len(b["q_off"])
    secs = []
    cb = None
    for i in range(args.warmup + args.steps):
        cb, _, cnt, t = cpu_reference_leg(b, full=True, repeats=1)
        if i >= args.warmup:
            secs.append(t)
    ms = 1e3 * float(np.mean(secs))
    v = n / (ms * 1e-3)
    cb["value"] = v
    cb["per_core"] = v / cb["cores"]
    cb["sample"] = f"all {n} jobs of the step batch per step, {args.steps} timed steps after {args.warmup} warm-up steps, on {cb['cores']} threads"
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u64 bit-vector (edlib)", "data": "synthetic",
        "config": workload_config(n),
        "cpu_baseline": cb, "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def pipeline_section(world, rank, local, dist):
    """Pipeline-level runs through the product binding (BAM + FASTA in, BCF out). N = 1: `delly_b200 sr` next to the reference's own drivers
    (oracle/_ref/delly_ref, all host threads), discovery and genotyping mode, BCFs compared byte for byte. N > 1: the SAME sample through N
    rank processes (one per GPU; scan + clustering replicated, assembly and genotyping sharded by SV range, ONE NCCL all-gatherv of the finished
    records per stage) — strong scaling; rank 0 then repeats the run single-rank and the two BCFs must be identical."""
    import subprocess
    import tempfile
    from delly_b200 import pipeline_bench as pb
    # N = 1 runs next to the reference's own drivers (6.5 s per run at 8 Mbp); N > 1 compares with a single-rank run of the binding only and takes a
    # sample three times the size, so that the fixed start-up (CUDA context, NCCL communicator) weighs less against the sharded stages
    glen, nsv, contigs = (8_000_000, 1600, 4) if world == 1 else (24_000_000, 4800, 8)
    out = {"config": {"workload": "configs[3]/[4]-shaped, scaled to fit the bench budget: synthetic 30x sample, 150 bp pairs, %d Mbp in %d contigs, %d planted "
                                  "het/hom DEL / DUP / INV" % (glen // 1_000_000, contigs, nsv), "scaling": "strong"}}
    if world > 1:
        box = [None]
        if rank == 0:
            box[0] = tempfile.mkdtemp(prefix="dgpu_pipe")
        dist.broadcast_object_list(box, src=0)
        d = box[0]
    else:
        d = tempfile.mkdtemp(prefix="dgpu_pipe")
    pre = os.path.join(d, "s")
    cores = host_cores()
    if rank == 0:
        out["simulate"] = pb.simulate(pre, glen, contigs, nsv, seed=11, threads=min(cores, 16))
    if world > 1:
        dist.barrier()
    res = {}
    if world > 1:
        # first the long-read chain over the same ranks: the reference's example/lr.bam (oracle/_ref/example travels with the repo), N ranks vs one rank.
        # It is tiny, so it also takes the one-off cost of the first communicator among fresh processes on a cold box off the timed runs below.
        ex = os.path.join(os.path.dirname(os.path.abspath(__file__)), "oracle", "_ref", "example")
        exe = os.path.join(pb.BIN, "delly_b200")
        if os.path.exists(os.path.join(ex, "lr.bam")):
            our = pre + f".lr.n{world}.bcf"
            cmd = [exe, "lr", "-g", os.path.join(ex, "ref.fa"), "-o", our, "--device", str(local), "--rank", str(rank), "--nranks", str(world),
                   "--comm-file", pre + ".lr.ncclid", os.path.join(ex, "lr.bam")]
            dist.barrier()
            t0 = time.perf_counter()
            r = subprocess.run(cmd, capture_output=True, text=True)
            dt = time.perf_counter() - t0
            if r.returncode != 0:
                raise RuntimeError(f"rank {rank}: delly_b200 lr failed: " + r.stderr[-600:])
            if rank == 0:
                one = pre + ".lr.n1.bcf"
                t1 = time.perf_counter()
                r1 = subprocess.run([exe, "lr", "-g", os.path.join(ex, "ref.fa"), "-o", one, "--device", str(local), os.path.join(ex, "lr.bam")], capture_output=True, text=True)
                t1 = time.perf_counter() - t1
                res["lr_example"] = {"wall_s_rank0": dt, "single_rank_s": t1, "bcf_identical_to_single_rank": r1.returncode == 0 and pb.inflate(one) == pb.inflate(our),
                                     "records": pb.count_records(our), "note": "reference fixture example/lr.bam (tiny): a correctness run of the sharded long-read chain over NCCL"}
            dist.barrier()
    for mode in ("discovery", "genotyping_mode"):
        sites = (pre + ".sites.bcf") if mode == "genotyping_mode" else None
        if world == 1:
            our, ref = pre + f".{mode}.ours.bcf", pre + f".{mode}.ref.bcf"
            pb.run_ours(pre, our, device=local, sites=sites)                                   # warm-up: page cache, CUDA module load
            runs = [pb.run_ours(pre, our, device=local, sites=sites, timing=pre + f".{mode}.json") for _ in range(2)]   # best of two (shared host)
            t_ours, stages = min(runs, key=lambda r: r[0])
            t_ref = pb.run_reference(pre, ref, threads=cores, sites=sites)
            res[mode] = {"ours_s": t_ours, "ours_runs_s": [r[0] for r in runs], "reference_s": t_ref, "speedup": t_ref / t_ours, "reference_threads": cores,
                         "bcf_identical": pb.inflate(ref) == pb.inflate(our), "records": pb.count_records(ref),
                         "stages_ms": stages["stages_ms"] if stages else None, "process_overhead_s": t_ours - (stages["total_ms"] * 1e-3 if stages else 0)}
            if mode == "discovery":
                os.replace(ref, pre + ".sites.bcf")
                if os.path.exists(ref + ".csi"):
                    os.replace(ref + ".csi", pre + ".sites.bcf.csi")
        else:
            if mode == "genotyping_mode" and rank == 0 and not os.path.exists(pre + ".sites.bcf"):
                raise RuntimeError("site list missing")
            comm_file = pre + f".{mode}.ncclid"
            our = pre + f".{mode}.n{world}.bcf"
            dist.barrier()
            t0 = time.perf_counter()
            r = subprocess.run(pb.ours_cmd(pre, our, device=local, sites=sites, rank=rank, nranks=world, comm_file=comm_file, timing=pre + f".{mode}.t"),
                               capture_output=True, text=True)
            dt = time.perf_counter() - t0
            if r.returncode != 0:
                raise RuntimeError(f"rank {rank}: delly_b200 failed: " + r.stderr[-600:])
            import torch
            t = torch.tensor([dt], device=torch.device("cuda", local))
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            wall = float(t.item())
            if rank == 0:
                one = pre + f".{mode}.n1.bcf"
                t1, st1 = pb.run_ours(pre, one, device=local, sites=sites, timing=pre + f".{mode}.t1")
                stages = json.load(open(pre + f".{mode}.t.0"))
                res[mode] = {"wall_s_max_over_ranks": wall, "single_rank_s_same_box": t1, "speedup_vs_single_rank": t1 / wall,
                             "bcf_identical_to_single_rank": pb.inflate(one) == pb.inflate(our), "records": pb.count_records(our),
                             "stages_ms_rank0": stages["stages_ms"], "stages_ms_single_rank": st1["stages_ms"] if st1 else None}
                if mode == "discovery":
                    os.replace(one, pre + ".sites.bcf")
            dist.barrier()
    out.update(res)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--jobs", type=int, default=JOBS_PER_STEP)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-families", action="store_true")
    ap.add_argument("--no-pipeline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the edit distances of the last timed step to DIR/*.npy (float32, at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference_arm(args)

    import torch
    import delly_b200

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dist_on = world > 1
    torch.cuda.set_device(local)
    if dist_on:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    ctx = delly_b200.Context(local)
    ctx.set_profiling(True)

    # weak scaling: every rank realigns its own 10 M-job shard of reads (independent jobs, no data-path collective)
    b = make_batch(args.jobs, seed=1001 + 100 * rank)
    n = len(b["q_off"])
    ops, byts, cells = algorithmic_counts(b)
    names = ("seqs", "q_off", "q_len", "t_off", "t_len", "k")
    pinned = {k: torch.from_numpy(b[k]).pin_memory() for k in names}
    d_in = {k: pinned[k].to(dev, non_blocking=True) for k in names}
    d_dist = torch.empty(n, dtype=torch.int32, device=dev)
    h_dist = torch.empty(n, dtype=torch.int32).pin_memory()
    torch.cuda.synchronize()
    # a non-default torch stream: the library launches on it and torch's events time it
    tstream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(tstream)
    stream = tstream.cuda_stream
    assert stream != 0

    # N > 1: the path's one exchange — an all-gatherv of every rank's finished call records through the product entry point
    # dgpu_gather_records (NCCL C API, its own communicator created with dgpu_comm_init; the 128-byte id travels through torch.distributed).
    # It runs INSIDE the timed region, once per step, with a payload of the size a chr20-scale shard produces (~2000 SV records with
    # consensus and per-sample count vectors, ~1 KB each).
    comm = delly_b200.C.c_void_p(0)
    gctx = None
    payload = None
    if dist_on:
        lib = delly_b200.lib()
        idbuf = torch.zeros(128, dtype=torch.uint8)
        if rank == 0:
            raw = (delly_b200.C.c_uint8 * 128)()
            ctx.check(lib.dgpu_comm_unique_id(raw), "dgpu_comm_unique_id")
            idbuf = torch.tensor(list(raw), dtype=torch.uint8)
        idt = idbuf.to(dev)
        dist.broadcast(idt, src=0)
        idraw = (delly_b200.C.c_uint8 * 128)(*idt.cpu().tolist())
        gctx = delly_b200.Context(local)          # the exchange has its own context / stream (as the binding's gather has)
        ctx.check(lib.dgpu_comm_init(gctx.h, world, rank, idraw, delly_b200.C.byref(comm)), "dgpu_comm_init")
        payload = np.random.default_rng(7 + rank).integers(0, 256, size=2_000_000 + 1000 * rank, dtype=np.uint8)

    def gather_step(buf):
        allp, cnts, nr = delly_b200.C.c_void_p(), delly_b200.C.c_void_p(), delly_b200.C.c_int()
        ctx.check(lib.dgpu_gather_records(gctx.h, comm, delly_b200._ptr(buf), delly_b200.C.c_uint64(buf.nbytes), delly_b200.C.byref(allp), delly_b200.C.byref(cnts),
                                          delly_b200.C.byref(nr)), "dgpu_gather_records")
        assert nr.value == world
        c = np.ctypeslib.as_array(delly_b200.C.cast(cnts, delly_b200.C.POINTER(delly_b200.C.c_uint64)), shape=(world,)).copy()
        lib.dgpu_free_host(allp); lib.dgpu_free_host(cnts)
        return c

    def dev_step():
        ctx.edit_distance_dev(d_in["seqs"], d_in["q_off"], d_in["q_len"], d_in["t_off"], d_in["t_len"], d_in["k"],
                              delly_b200.MODE_HW, d_dist, None, stream)
        if dist_on:
            torch.cuda.current_stream().synchronize()      # the records of a step exist when its realignments are done
            gather_step(payload)

    def barrier():
        if dist_on:
            dist.barrier()
        torch.cuda.synchronize()

    # configs[1] jobs are probes of <= 80 bp against 150 bp reads: with the bound set the device form never synchronises (include/dgpu.h)
    ctx.check(delly_b200.lib().dgpu_set_async_bound(ctx.h, 256), "dgpu_set_async_bound")
    for _ in range(args.warmup):
        dev_step()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    l0 = ctx.launches
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    kern_ms = []
    barrier()
    ev0.record()
    for _ in range(args.steps):
        dev_step()
        kern_ms.append(None)
    ev1.record()
    barrier()
    total_ms = ev0.elapsed_time(ev1)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, d_dist.cpu().numpy(), world, rank)     # before the untimed runs below reuse d_dist
    launches = ctx.launches - l0
    # dominant-kernel span (library-side CUDA events on the launching stream), measured outside the loop timing
    kms = []
    for _ in range(max(3, args.steps)):
        dev_step()
        kms.append(ctx.last_kernel_ms())
    clocks = sampler.stop() if rank == 0 else None
    if dist_on:
        t = torch.tensor([total_ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms = float(t.item())
    ms_per_step = total_ms / args.steps
    value = world * n / (ms_per_step * 1e-3)

    ctx.check(delly_b200.lib().dgpu_set_async_bound(ctx.h, 0), "dgpu_set_async_bound")
    # end-to-end through the host-pointer ABI (pinned buffers; H2D of inputs and D2H of results inside the timed region)
    def e2e_step():
        rc = ctx._lib.dgpu_edit_distance(ctx.h, delly_b200._ptr(pinned["seqs"]), delly_b200.C.c_uint64(pinned["seqs"].numel()),
                                         delly_b200._ptr(pinned["q_off"]), delly_b200._ptr(pinned["q_len"]),
                                         delly_b200._ptr(pinned["t_off"]), delly_b200._ptr(pinned["t_len"]),
                                         delly_b200._ptr(pinned["k"]), delly_b200.MODE_HW, delly_b200.C.c_uint64(n),
                                         delly_b200._ptr(h_dist), delly_b200.C.c_void_p(0))
        ctx.check(rc, "dgpu_edit_distance")

    for _ in range(2):
        e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        e2e_step()
    barrier()
    e2e_s = time.perf_counter() - t0
    if dist_on:
        t = torch.tensor([e2e_s], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
    e2e_value = world * n * args.steps / e2e_s
    h2d = sum(pinned[k].numel() * pinned[k].element_size() for k in names)
    d2h = h_dist.numel() * 4
    # results of both paths must agree (and are spot-checked against the CPU leg below)
    assert torch.equal(h_dist, d_dist.cpu()), "device-resident and host-ABI results differ"

    gather_ms = gather_ms_50mb = None
    if dist_on:
        # the exchange on its own: (i) the per-step payload, (ii) a genome-scale payload (50 MB over all ranks, SURVEY section 8e upper bound)
        for _ in range(2):
            gather_step(payload)
        barrier(); t0 = time.perf_counter()
        for _ in range(5):
            cnts = gather_step(payload)
        gather_ms = (time.perf_counter() - t0) * 1e3 / 5
        assert int(cnts[rank]) == payload.nbytes and len(cnts) == world
        big = np.zeros(50_000_000 // world, np.uint8)
        gather_step(big)
        barrier(); t0 = time.perf_counter()
        for _ in range(3):
            gather_step(big)
        gather_ms_50mb = (time.perf_counter() - t0) * 1e3 / 3
        t = torch.tensor([gather_ms, gather_ms_50mb], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        gather_ms, gather_ms_50mb = float(t[0].item()), float(t[1].item())
    pipeline = None
    pipeline_error = None
    if not args.no_pipeline:
        try:
            pipeline = pipeline_section(world, rank, local, dist if dist_on else None)
        except Exception as e:  # noqa: BLE001  (auxiliary: the headline line must still print)
            pipeline_error = repr(e)
            if dist_on:
                pass
    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s"
        kmed = float(np.median(kms))
        tops = delly_b200.C.c_double(ctx.int_peak_tops())
        traffic = None
        try:  # DRAM bytes per job of the dominant kernels from the committed ncu --set full capture (profiles/)
            tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
            traffic = tj["ed_small_dram_bytes_per_job"] * n
        except Exception:
            pass
        ach_gbs = byts / (kmed * 1e-3) / 1e9
        ach_tops = ops / (kmed * 1e-3) / 1e12
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u32 bit-vector words (Myers), int32 scores", "data": "synthetic",
            "config": workload_config(n, world=world),
            "gpu_launches": launches,
            "gather_ms": gather_ms, "gather_ms_50mb_total_payload": gather_ms_50mb,
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            # the binding roof of this path is the integer pipe (about %d int32 ops per input byte); HBM figures ride along as secondary keys
            "roofline": {"bound": "int32 ALU", "achieved": ach_tops, "peak": tops.value, "unit": "Tint32op/s", "frac": ach_tops / tops.value,
                         "traffic": traffic, "peak_source": "measured live: dgpu_int_peak (8 independent LOP3 chains per thread; = 148 SMs x 64 lanes x clock); "
                                                            "MEASURED_PEAKS.json carries no integer figure", "int32_top_s": tops.value,
                         "kernel": "ed_small_kernel<NW,HW> (all NW classes of one step)", "kernel_ms": kmed, "algorithmic_ops_per_step": ops,
                         "gcups": cells / (kmed * 1e-3) / 1e9,
                         "hbm": {"achieved": ach_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": ach_gbs / hbm_peak, "peak_source": peak_src,
                                 "algorithmic_bytes_per_step": byts}},
        }
        if pipeline is not None:
            out["pipeline"] = pipeline
        if pipeline_error is not None:
            out["pipeline_error"] = pipeline_error
        if not args.no_cpu and world == 1:
            cb, cd, cnt, _t = cpu_reference_leg(b)
            assert np.array_equal(cd, h_dist.numpy()[:cnt]), "GPU results differ from the CPU reference on the sample"
            out["cpu_baseline"] = cb
        if not args.no_families and world == 1:
            try:
                out["families"] = bench_families(ctx)
            except Exception as e:  # noqa: BLE001  (the headline line must still print)
                out["families_error"] = repr(e)
        print(json.dumps(out))
    if dist_on:
        lib.dgpu_comm_destroy(gctx.h, comm)
        gctx.close()
        dist.destroy_process_group()
    ctx.close()


if __name__ == "__main__":
    main()
