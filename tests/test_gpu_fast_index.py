"""GPU parity of the single-population fast path's key-only index of the full haplotypes (FastIndex,
csrc/grimb_tables.h) against the CPU oracle:
- a zipf table with the index at 2 slots per haplotype (GRIMB_FAST_INDEX_MULT=2: half full, so many
  sectors carry the overflow flag and probes scan past their home sector) and at the default size;
- a table of eight haplotypes in four sectors, picked with the hash so that six share the last
  sector: flagged misses, hits past the home sector and the wrap-around to sector 0 are certain;
- a table restored from its device image (grimb_tables_from_image rebuilds the index) gives the
  same output as the table it was copied from.
Subjects with more than four candidate phases (the long form) are covered by test_gpu_split_path.py."""
import itertools
import json
import os

import numpy as np
import pytest

import goldenlib
import grim_oracle as go
import synth
from emu_backend import hash_key

pytestmark = pytest.mark.gpu

LOCI = ["A", "B", "C", "DQB1", "DRB1"]


def _conf(d, hpf, over=None):
    open(d + "/hpf.csv", "w").write(hpf)
    open(d + "/cnt.txt", "w").write("CAU,1000.0,1.0\n")
    conf = json.load(open(os.path.join(goldenlib.GOLD, "data", "base_conf.json")))
    conf.update({"freq_file": d + "/hpf.csv", "pops_count_file": d + "/cnt.txt", "freq_trim_threshold": 1e-30})
    conf.update(over or {})
    return conf


def _run(conf, lines, graph=None):
    """-> (output texts, graph) through the CUDA path; asserts that the split fast path ran."""
    from grim.imputation.impute import Imputation
    from grim.imputation.networkx_graph import Graph
    from grim.run_impute_def import load_config
    cfg = load_config(conf)
    g = graph if graph is not None else Graph(cfg).build_graph()
    imp = Imputation(g, cfg)
    out = imp.impute_text("".join(lines).encode("utf8"))
    assert g.lib.grimb_engine_kernel_ms(g.engine(imp.workspaces[0]), 4) >= 0, "the split fast path did not run"
    return {k: out[k].decode("utf8") for k in goldenlib.KEYS}, g


def _check(conf, lines, out):
    ref, _ = go.impute_file(conf, lines=lines)
    for k in goldenlib.KEYS:
        assert out[k] == ref[k], "%s differs from the oracle" % k


@pytest.mark.parametrize("mult", ["2", None])
def test_fast_index_zipf_table(mult, tmp_path, monkeypatch):
    monkeypatch.setenv("GRIMB_HOST_EVENTS", "1")   # kernel timing events in the host-pointer path
    if mult is None:
        monkeypatch.delenv("GRIMB_FAST_INDEX_MULT", raising=False)
    else:
        monkeypatch.setenv("GRIMB_FAST_INDEX_MULT", mult)   # read when the table is built
    hpf = synth.zipf_table(3000, [12, 20, 10, 6, 14], 5)
    conf = _conf(str(tmp_path), hpf)
    tab = synth.Table(hpf)
    lines = synth.typed_subjects(tab, 3000, 6, ["CAU,CAU"]) + synth.messy_subjects(tab, 100, 7)
    out, g = _run(conf, lines)
    _check(conf, lines, out)
    g.close()


def _colliding_table():
    """Eight haplotypes over three alleles per locus whose ids, packed as the library packs them, put six
    homes in sector 3 of a four-sector index (8 keys x 2 slots = 16 slots); every allele appears."""
    from grim.imputation.networkx_graph import key_layout
    names = [["%s*%02d:01" % (l, a + 1) for a in range(3)] for l in LOCI]
    bits = key_layout([3] * 5)
    shift = [int(sum(bits[:l])) for l in range(5)]
    haps = list(itertools.product(range(3), repeat=5))
    home = {h: hash_key(sum((a + 1) << shift[l] for l, a in enumerate(h))) & 3 for h in haps}
    rng = np.random.RandomState(11)
    last = [h for h in haps if home[h] == 3]
    rest = [h for h in haps if home[h] != 3]
    for _ in range(10000):
        pick = [last[i] for i in rng.choice(len(last), 6, replace=False)] + \
               [rest[i] for i in rng.choice(len(rest), 2, replace=False)]
        if all(len({h[l] for h in pick}) == 3 for l in range(5)):
            break
    else:
        raise AssertionError("no haplotype set with every allele")
    f = rng.lognormal(0.0, 1.0, size=len(pick))
    f /= f.sum()
    rows = ["hap,pop,freq\n"] + ["%s,CAU,%r\n" % ("~".join(names[l][a] for l, a in enumerate(h)), float(x))
                                 for h, x in zip(pick, f)]
    return names, pick, shift, "".join(rows)


def test_fast_index_shared_home_sectors(tmp_path, monkeypatch):
    monkeypatch.setenv("GRIMB_HOST_EVENTS", "1")
    monkeypatch.setenv("GRIMB_FAST_INDEX_MULT", "2")
    names, pick, shift, hpf = _colliding_table()
    conf = _conf(str(tmp_path), hpf)
    rng = np.random.RandomState(12)
    lines = []
    for s in range(2000):
        # half the subjects carry two haplotypes of the table (hits, some past their home sector); the rest
        # random alleles (misses, many in the flagged sector 3)
        if s % 2 == 0:
            h1, h2 = (pick[i] for i in rng.randint(0, len(pick), size=2))
        else:
            h1, h2 = rng.randint(0, 3, size=5), rng.randint(0, 3, size=5)
        sides = ["%s+%s" % (names[l][h1[l]], names[l][h2[l]]) for l in range(5)]
        lines.append("Q%d,%s,CAU,CAU\n" % (s, "^".join(sides)))
    out, g = _run(conf, lines)
    assert list(g.shift) == shift, "the library packs keys differently from this test"
    assert g.info()["n_full"] == 8
    _check(conf, lines, out)
    g.close()


def test_fast_index_from_image(tmp_path, monkeypatch):
    monkeypatch.setenv("GRIMB_HOST_EVENTS", "1")
    from grim.imputation.networkx_graph import Graph
    from grim.run_impute_def import load_config
    hpf = synth.zipf_table(2000, [10, 16, 8, 6, 12], 8)
    conf = _conf(str(tmp_path), hpf)
    tab = synth.Table(hpf)
    lines = synth.typed_subjects(tab, 2000, 9, ["CAU,CAU"])
    out1, g1 = _run(conf, lines)
    img = g1.image_to_host()
    g2 = Graph(load_config(conf)).from_image_host(img, g1.alleles)
    assert g2.info()["device_bytes"] == g1.info()["device_bytes"] > img.nbytes   # the index is not in the image
    out2, g2 = _run(conf, lines, graph=g2)
    assert out2 == out1
    g1.close()
    g2.close()
