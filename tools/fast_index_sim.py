"""fast_index_sim.py -- CPU model of the fast path's key-only full-haplotype index (FastIndex,
csrc/grimb_tables.h): 8-byte keys, four to a 32-byte sector, home sector hash_key(key) & mask, linear
probing by sector, optional per-sector overflow flag.  On bench.py's table and subjects (the library's
own key layout and hash; keys inserted in node order; every one of a subject's 32 haplotypes probed) it
reports the sectors read per probe and the share of warps (two subjects, 64 probes) whose slowest probe
needs two or three dependent sector trips.  Design aid for DESIGN.md sections 4 and 8; nothing here runs
on the product path, and no number it prints is a GPU measurement.

    python tools/fast_index_sim.py [--mult 4] [--no-flag] [--small]
"""
import argparse
import os
import sys

import numpy as np

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "py-graph-imputation_b200"))
import bench  # noqa: E402
from grim.imputation.networkx_graph import key_layout  # noqa: E402

M32 = np.uint64(0xFFFFFFFF)


def hash_key(k):
    """grimb_group.h hash_key() for 64-bit keys, vectorised."""
    h = (k & M32) ^ (((k >> np.uint64(32)) * np.uint64(0x9E3779B1)) & M32)
    h ^= h >> np.uint64(16)
    h = (h * np.uint64(0x85ebca6b)) & M32
    h ^= h >> np.uint64(13)
    h = (h * np.uint64(0xc2b2ae35)) & M32
    h ^= h >> np.uint64(16)
    return h.astype(np.int64)


def pack(al, shift):
    k = np.zeros(al.shape[0], np.uint64)
    for l in range(al.shape[1]):
        k |= al[:, l].astype(np.uint64) << np.uint64(shift[l])
    return k


def simulate(keys, probes, n_sectors, flag):
    """-> sectors read by each probe (probes: [S][32] keys)."""
    mask = n_sectors - 1
    fill = np.zeros(n_sectors, np.int64)         # keys stored per sector
    ovf = np.zeros(n_sectors, bool)
    where = {}
    home = hash_key(keys) & mask
    for k, h in zip(keys.tolist(), home.tolist()):
        s = h
        while fill[s] == 4:
            s = (s + 1) & mask
        fill[s] += 1
        where[k] = s
        if s != h:
            ovf[h] = True
    # sectors until one with an empty slot, from every sector on (cyclic)
    free = np.where(fill < 4)[0]
    idx = np.searchsorted(free, np.arange(n_sectors))
    nxt = np.where(idx < len(free), free[np.minimum(idx, len(free) - 1)], free[0] + n_sectors)
    scan = nxt - np.arange(n_sectors) + 1
    flat = probes.reshape(-1)
    ph = hash_key(flat) & mask
    miss = scan[ph] if not flag else np.where(ovf[ph], scan[ph], 1)
    sec = miss.astype(np.int64)
    for j, k in enumerate(flat.tolist()):
        s = where.get(k)
        if s is not None:
            sec[j] = ((s - ph[j]) & mask) + 1
    return sec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--mult", type=int, default=4, help="slots per full haplotype (GRIMB_FAST_INDEX_MULT)")
    ap.add_argument("--no-flag", action="store_true", help="no overflow flag: a miss scans to an empty slot")
    ap.add_argument("--small", action="store_true", help="100,000 haplotypes and 8,192 subjects (quick run)")
    a = ap.parse_args()
    n_full, n_subj = (100_000, 8192) if a.small else (1_000_000, 65536)
    _names, fa, ff = bench.make_table(n_full)
    bits = key_layout(bench.N_ALLELES)
    shift = [int(sum(bits[:l])) for l in range(5)]
    keys = pack(fa, shift)[ff[:, 0] > 0]
    _batch, al = bench.make_subjects(fa, ff, n_subj, bench.SUBJECT_SEED)
    probes = np.stack([pack(np.where(np.array([(m >> l) & 1 for l in range(5)], bool), al[:, :, 1], al[:, :, 0]), shift)
                       for m in range(32)], axis=1)
    n_slots = 4
    while n_slots < a.mult * len(keys):
        n_slots <<= 1
    sec = simulate(keys, probes, n_slots // 4, not a.no_flag)
    warp = sec.reshape(-1, 64).max(axis=1)
    print("haplotypes %d  subjects %d  index %d MB keys (mult %d, flag %s)" %
          (len(keys), n_subj, n_slots * 8 >> 20, a.mult, "off" if a.no_flag else "on"))
    print("sectors/probe %.4f  warps needing >= 2 trips %.4f  >= 3 trips %.4f" %
          (sec.mean(), (warp >= 2).mean(), (warp >= 3).mean()))


if __name__ == "__main__":
    main()
