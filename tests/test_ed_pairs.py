"""HW realign pairs (two probes against the same read in one thread) and the top-aligned HW distance kernel, against the oracle.

Jobs 2j and 2j+1 share a thread when both are thread-per-job HW jobs over the same target bytes (equal t_off and t_len) and no end
locations are asked for. The batches here hit every edge of that rule: probe lengths on both sides of the 32-row word boundaries, members
of one pair in different word classes, targets shorter than or not a multiple of the 16-byte chunk, odd job counts, broken pairs, bytes
outside ACGTN, bounds k that turn answers into -1, shuffled orders, and the modes and end-location calls that must keep their old path."""
import numpy as np
import pytest

from delly_b200 import synth
from oracle import pyoracle as po

ALPHA = np.frombuffer(b"ACGT", np.uint8)
QLENS = [1, 31, 32, 33, 63, 64, 65, 96, 97, 127, 128]
TLENS = [1, 3, 15, 16, 17, 31, 33, 47, 150, 151, 200]
WEIRD = np.frombuffer(b"NNRYacgtn-", np.uint8)


def _probe(rng, t, ql):
    """A probe of ql bytes: mostly a noisy piece of the read (so that distances are small), sometimes random."""
    if len(t) > 4 and rng.random() < 0.7:
        a = int(rng.integers(0, max(1, len(t) - ql // 2)))
        q = np.resize(t[a:a + ql], ql).copy()
        q = synth.mutate(rng, q, sub=0.03, ins=0.02, dele=0.02)
        q = np.resize(q, ql) if len(q) else ALPHA[rng.integers(0, 4, size=ql)]
        return q.astype(np.uint8)
    return ALPHA[rng.integers(0, 4, size=ql)]


def _sprinkle(rng, arr):
    arr = arr.copy()
    for p in rng.integers(0, len(arr), size=max(1, len(arr) // 12)):
        arr[p] = rng.choice(WEIRD)
    return arr


def _pair_batch(seed, n_reads, weird=0.0, broken=0.0, equal=0.3, odd=False):
    """n_reads reads, each with an (ALT, REF)-like probe pair at jobs 2i, 2i+1 over the same read bytes. `broken` of the pairs point the
    second job at a byte-identical copy of the read (equal t_len, different t_off); `weird` of the sequences carry bytes outside ACGT."""
    rng = np.random.default_rng(seed)
    seqs, spec = [], []
    for i in range(n_reads):
        tl = int(rng.choice(TLENS)) if rng.random() < 0.5 else int(rng.integers(1, 260))
        t = ALPHA[rng.integers(0, 4, size=tl)]
        la = int(rng.choice(QLENS)) if rng.random() < 0.6 else int(rng.integers(1, 129))
        lb = la if rng.random() < equal else (int(rng.choice(QLENS)) if rng.random() < 0.6 else int(rng.integers(1, 129)))
        qa, qb = _probe(rng, t, la), _probe(rng, t, lb)
        if rng.random() < weird:
            t = _sprinkle(rng, t)
        if rng.random() < weird:
            qa = _sprinkle(rng, qa)
        if rng.random() < weird:
            qb = _sprinkle(rng, qb)
        base = len(seqs)
        seqs += [qa, qb, t]
        tb = base + 2
        if rng.random() < broken:
            seqs.append(t.copy())
            tb = base + 3
        spec.append((base, base + 1, base + 2, tb))
    arena, off, ln = synth.pack(seqs)
    q_idx = np.array([[a, b] for a, b, _, _ in spec]).reshape(-1)
    t_idx = np.array([[ta, tb] for _, _, ta, tb in spec]).reshape(-1)
    b = dict(seqs=arena, q_off=off[q_idx].copy(), q_len=ln[q_idx].copy(), t_off=off[t_idx].copy(), t_len=ln[t_idx].copy())
    n = len(b["q_off"]) - (1 if odd else 0)
    for key in ("q_off", "q_len", "t_off", "t_len"):
        b[key] = np.ascontiguousarray(b[key][:n])
    kc = rng.integers(0, 4, size=n)
    b["k"] = np.where(kc == 0, -1, np.where(kc == 1, rng.integers(0, 4, size=n),
                      np.where(kc == 2, synth.hw_k(b["q_len"]), 10 ** 6))).astype(np.int32)
    return b


def _sub(b, idx):
    return {k: (v if k == "seqs" else np.ascontiguousarray(v[idx])) for k, v in b.items()}


def _oracle(b, mode=2, want_end=False):
    d, e = po.edit_distance_batch(po.oracle(), b["seqs"], b["q_off"], b["q_len"], b["t_off"], b["t_len"], b["k"], mode,
                                  threads=8, want_end=True)
    return (d, e) if want_end else d


def _paired_fraction(b):
    """Share of the jobs the pairing rule puts into pairs (the tests must exercise the pair path, not only the single one)."""
    n = len(b["q_off"]) // 2 * 2
    ev, od = np.arange(0, n, 2), np.arange(1, n, 2)
    ok = ((b["t_off"][ev] == b["t_off"][od]) & (b["t_len"][ev] == b["t_len"][od]) & (b["t_len"][ev] > 0)
          & (b["q_len"][ev] >= 1) & (b["q_len"][ev] <= 128) & (b["q_len"][od] >= 1) & (b["q_len"][od] <= 128))
    return 2 * ok.sum() / max(1, len(b["q_off"]))


def _dev(ctx, b, mode=2, stream=None):
    import torch
    dev = torch.device("cuda", 0)
    t = {k: torch.from_numpy(np.ascontiguousarray(b[k])).to(dev) for k in ("seqs", "q_off", "q_len", "t_off", "t_len", "k")}
    out = torch.full((len(b["q_off"]),), -7, dtype=torch.int32, device=dev)
    ctx.edit_distance_dev(t["seqs"], t["q_off"], t["q_len"], t["t_off"], t["t_len"], t["k"], mode, out, None, stream)
    torch.cuda.synchronize()
    return out.cpu().numpy()


def _async(ctx, b, mode=2):
    assert ctx._lib.dgpu_set_async_bound(ctx.h, 256) == 0
    try:
        return _dev(ctx, b, mode)
    finally:
        ctx._lib.dgpu_set_async_bound(ctx.h, 0)


def _check(got, want, b, what):
    bad = np.nonzero(got != want)[0]
    assert len(bad) == 0, (what, bad[:6], got[bad[:6]], want[bad[:6]], b["q_len"][bad[:6]], b["t_len"][bad[:6]], b["k"][bad[:6]])


def test_pair_batches_exercise_the_pair_rule():
    b = _pair_batch(1, 400, broken=0.2)
    f = _paired_fraction(b)
    assert 0.6 < f < 0.95
    qa, qb = b["q_len"][0::2], b["q_len"][1::2]
    assert np.any((qa + 31) // 32 != (qb + 31) // 32) and np.any(qa == qb)
    assert _paired_fraction(_pair_batch(2, 50, odd=True)) < 1.0


@pytest.mark.gpu
@pytest.mark.parametrize("form", ["host", "device", "async"])
@pytest.mark.parametrize("case", ["plain", "weird", "broken_odd"])
def test_pairs_match_oracle(ctx, form, case):
    kw = {"plain": {}, "weird": {"weird": 0.4}, "broken_odd": {"broken": 0.3, "odd": True}}[case]
    b = _pair_batch(100 + len(case) + len(form), 3000, **kw)
    want = _oracle(b)
    if form == "host":
        got = ctx.edit_distance(b["seqs"], b["q_off"], b["q_len"], b["t_off"], b["t_len"], b["k"], 2)
    elif form == "device":
        got = _dev(ctx, b)
    else:
        got = _async(ctx, b)
    _check(got, want, b, (form, case))
    assert np.any(want == -1) and np.any(want == 0)


@pytest.mark.gpu
def test_every_length_pairing(ctx):
    """Every (|qA|, |qB|) over the word-boundary lengths, against targets from 1 to 200 bytes, both members noisy copies of the read."""
    rng = np.random.default_rng(7)
    seqs, qi, ti = [], [], []
    for la in QLENS:
        for lb in QLENS:
            for tl in (1, 7, 16, 31, 150, 200):
                t = ALPHA[rng.integers(0, 4, size=tl)]
                s = len(seqs)
                seqs += [_probe(rng, t, la), _probe(rng, t, lb), t]
                qi += [s, s + 1]
                ti += [s + 2, s + 2]
    arena, off, ln = synth.pack(seqs)
    qi, ti = np.array(qi), np.array(ti)
    b = dict(seqs=arena, q_off=off[qi].copy(), q_len=ln[qi].copy(), t_off=off[ti].copy(), t_len=ln[ti].copy())
    b["k"] = np.full(len(qi), -1, np.int32)
    want = _oracle(b)
    _check(ctx.edit_distance(b["seqs"], b["q_off"], b["q_len"], b["t_off"], b["t_len"], b["k"], 2), want, b, "host")
    _check(_async(ctx, b), want, b, "async")


@pytest.mark.gpu
def test_shuffled_order_and_other_paths(ctx):
    """A shuffled job order (pairs mostly broken), and on the same batch the NW / SHW modes and HW with end locations (never paired)."""
    b = _pair_batch(31, 2500, weird=0.2, broken=0.1)
    want = _oracle(b)
    perm = np.random.default_rng(3).permutation(len(want))
    s = _sub(b, perm)
    _check(ctx.edit_distance(s["seqs"], s["q_off"], s["q_len"], s["t_off"], s["t_len"], s["k"], 2), want[perm], s, "shuffled")
    _check(_async(ctx, s), want[perm], s, "shuffled async")
    for mode in (0, 1, 2):
        d, e = _oracle(b, mode, want_end=True)
        gd, ge = ctx.edit_distance(b["seqs"], b["q_off"], b["q_len"], b["t_off"], b["t_len"], b["k"], mode, want_end=True)
        _check(gd, d, b, ("end", mode))
        ok = d >= 0
        assert np.array_equal(ge[ok], e[ok]) and np.all(ge[~ok] == -1)
        if mode != 2:
            _check(ctx.edit_distance(b["seqs"], b["q_off"], b["q_len"], b["t_off"], b["t_len"], b["k"], mode), d, b, ("dist", mode))


@pytest.mark.gpu
def test_k1_shape_with_unequal_probes(ctx):
    """K1 batch (probe pairs over shared reads) with the REF probe shortened by 0-40 bytes: pairs whose members differ in length and class."""
    b = synth.k1_genotype_batch(200_001, seed=91)
    rng = np.random.default_rng(4)
    cut = rng.integers(0, 41, size=len(b["q_len"]) // 2 + 1)[: (len(b["q_len"]) + 1) // 2]
    ql = b["q_len"].astype(np.int64)
    ql[1::2] = np.maximum(1, ql[1::2] - cut[: len(ql[1::2])])
    b["q_len"] = ql.astype(np.uint32)
    b["k"] = synth.hw_k(b["q_len"])
    sel = np.concatenate([np.arange(0, 4000), np.arange(len(ql) - 2001, len(ql))])
    got = _async(ctx, b)
    got_host = ctx.edit_distance(b["seqs"], b["q_off"], b["q_len"], b["t_off"], b["t_len"], b["k"], 2)
    assert np.array_equal(got, got_host)
    s = _sub(b, sel)
    _check(got[sel], _oracle(s), s, "k1 sample")
