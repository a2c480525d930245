"""CPU model of k_fast_probe2's queue (csrc/grimb200.cu): replays its enqueue and drain policy warp by warp on
bench.py's C2 batch and on adversarial batches, and reports the probes per subject at each level, the drains
per loop iteration and the peak queue fill, asserted against the bound argued in the kernel (<= 110 of 128).

Policy, as the kernel runs it: warp w takes subjects s0 .. s0+3 per iteration (s0 = 4 w, 4 (w + nw), ...);
  1. a queue holding >= 32 entries is drained once, with the iteration's level-1 loads in flight;
  2. each heterozygous subject appends one entry per level-1 hit (its entries contiguous);
  3. while the queue holds >= 64 entries it is drained again (no overlap);
  after the loop, drains until empty.  A drain takes the whole subjects among the first 32 entries.
Level 1 probes phase i's first haplotype when the phase is kept and neither side holds an unknown allele;
the one-level kernel probes both haplotypes of every kept phase whose side is known.

  python tools/probe_queue_sim.py [--subjects N] [--haps N] [--sms 148] [--ctas 4]"""
import argparse
import itertools
import os
import sys
from collections import deque

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

CAP, DRAIN, HIGH = 128, 32, 64


def phase_probes(alleles, table_keys, n_alleles):
    """alleles [S][5][2] (1-based) -> (eligible [S][16], hit1 [S][16], old probes per subject, same [S]).
    hit1: the first haplotype is in the table (only where eligible)."""
    S, L = alleles.shape[0], alleles.shape[1]
    het = (alleles[:, :, 0] != alleles[:, :, 1])
    hm = (het * (1 << np.arange(L))).sum(axis=1)
    unk = alleles > np.asarray(n_alleles)[None, :, None]          # [S][L][2]
    low = hm & ((1 << (L - 1)) - 1)
    last_het = (hm >> (L - 1)) & 1
    eligible = np.zeros((S, 16), bool)
    hit1 = np.zeros((S, 16), bool)
    old = np.zeros(S)
    for i in range(1 << (L - 1)):
        side = np.array([(i >> l) & 1 for l in range(L)])          # side of haplotype 1 at each locus
        kept = ((i & ~low) == 0) & ((last_het == 1) | (i <= (low ^ i)))
        known1 = ~unk[:, np.arange(L), side].any(axis=1)
        known2 = ~unk[:, np.arange(L), 1 - side].any(axis=1)
        key1 = np.zeros(S, np.int64)
        for l in range(L):
            key1 = key1 * 4096 + alleles[:, l, side[l]]
        eligible[:, i] = kept & known1 & known2
        hit1[:, i] = eligible[:, i] & np.isin(key1, table_keys)
        old += kept * (known1.astype(int) + known2.astype(int))
    return eligible, hit1, old, hm == 0


def simulate(eligible, hit1, same, n_warps):
    """-> dict of per-subject / per-iteration figures of the queue policy."""
    S = len(same)
    entries = np.where(same, 0, hit1.sum(axis=1))
    stride = n_warps * 4
    it = drains_ov = drains_extra = drains_flush = 0
    peak = 0
    for w in range(n_warps):
        q = deque()   # entry counts of the queued subjects, in order
        qn = 0

        def drain():
            nonlocal qn
            taken = 0
            while q and taken + q[0] <= DRAIN:
                taken += q.popleft()
            assert taken >= (DRAIN // 2 + 1 if qn > DRAIN else qn), "a drain must take >= 17 entries or all"
            qn -= taken

        for s0 in range(4 * w, S, stride):
            it += 1
            if qn >= DRAIN:
                drain()
                drains_ov += 1
            for s in range(s0, min(s0 + 4, S)):
                if entries[s]:
                    q.append(int(entries[s]))
                    qn += int(entries[s])
            peak = max(peak, qn)
            assert qn <= 110 <= CAP, "queue bound violated: %d" % qn
            while qn >= HIGH:
                drain()
                drains_extra += 1
        while qn > 0:
            drain()
            drains_flush += 1
    return {"iterations": it, "drains_overlapped_per_iteration": drains_ov / max(it, 1),
            "drains_extra_per_iteration": drains_extra / max(it, 1), "drains_flush_per_warp": drains_flush / n_warps,
            "peak_queue_entries": peak, "level2_probes_per_subject": float(entries.mean()),
            "same_subjects": float(same.mean())}


def report(name, alleles, table_keys, n_alleles, n_warps):
    eligible, hit1, old, same = phase_probes(alleles, table_keys, n_alleles)
    r = simulate(eligible, hit1, same, n_warps)
    l1 = float(eligible.sum(axis=1).mean())
    print("%s: subjects %d, one-level probes/subject %.2f, level-1 %.2f, level-2 %.2f, two-level total %.2f (%.1f %% fewer); "
          "level-1 hits/subject %.2f; drains/iteration %.3f overlapped + %.3f extra, flush %.2f/warp; peak queue %d of %d"
          % (name, len(same), old.mean(), l1, r["level2_probes_per_subject"], l1 + r["level2_probes_per_subject"],
             100 * (1 - (l1 + r["level2_probes_per_subject"]) / old.mean()), float(hit1.sum(axis=1).mean()),
             r["drains_overlapped_per_iteration"], r["drains_extra_per_iteration"], r["drains_flush_per_warp"],
             r["peak_queue_entries"], CAP))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--subjects", type=int, default=1 << 20)
    ap.add_argument("--haps", type=int, default=1000000)
    ap.add_argument("--sms", type=int, default=148)
    ap.add_argument("--ctas", type=int, default=4, help="resident CTAs per SM (FASTPROBE2_MIN_BLOCKS)")
    a = ap.parse_args()
    import bench
    n_warps = a.sms * a.ctas * 8
    names, fa, ff = bench.make_table(a.haps)
    n_alleles = [len(x) for x in names]
    tk = np.zeros(len(fa), np.int64)
    for l in range(5):
        tk = tk * 4096 + fa[:, l]
    _b, alleles = bench.make_subjects(fa, ff, a.subjects, bench.SUBJECT_SEED)
    print("warps %d (%d SMs x %d CTAs x 8)" % (n_warps, a.sms, a.ctas))
    report("bench C2", alleles.astype(np.int64), tk, n_alleles, n_warps)
    # adversarial: a table of every 0/1 haplotype and subjects 0/1 at every locus -> 16 level-1 hits each
    two = np.array(list(itertools.product((1, 2), repeat=5)), np.int64)
    tk2 = np.zeros(len(two), np.int64)
    for l in range(5):
        tk2 = tk2 * 4096 + two[:, l]
    S2 = 1 << 16
    adv = np.zeros((S2, 5, 2), np.int64)
    adv[:, :, 0], adv[:, :, 1] = 1, 2
    report("all 16 phases hit", adv, tk2, [2] * 5, n_warps)
    rng = np.random.RandomState(5)
    mix = rng.randint(1, 3, size=(S2, 5, 2)).astype(np.int64)
    report("random 0/1 subjects", mix, tk2, [2] * 5, n_warps)
    half = adv.copy()
    half[::3] = mix[::3]
    half[1::7, 2, 1] = 3       # an unknown allele on one side
    report("mixed with unknown alleles", half, tk2, [2] * 5, n_warps)


if __name__ == "__main__":
    main()
