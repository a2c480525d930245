"""GPU: the two-level probe kernel of the split fast path (k_fast_probe2: level 1 probes a phase's first
haplotype, a per-warp queue collects the hits, level 2 probes their second haplotypes 32 at a time) against
the one-level k_fast_probe (GRIMB_FAST_PROBE=1) and the CPU oracle.  Every case compares the six files and the
pair-evaluation count of both kernels with the oracle's.  The cases aim at the queue: subjects with many
level-1 hits and no candidate (16 entries per subject, so the queue fills past its drain threshold and drains
cut inside a subject's entries), more candidate phases than a hand-over record holds and the exhaustion of the
side records, homozygous subjects, unknown alleles, four loci, a batch that is not a multiple of the four
subjects a warp takes, chunked host calls (a non-zero first subject), colliding index sectors and the general
batch form (which keeps the one-level kernel).  Each arm asserts which probe kernel ran and on which batch form,
and that both handed the same number of subjects to the general kernel.  One case, too large for the oracle,
compares the two kernels on a batch big enough that every warp runs several iterations with a well-filled
queue (overlapped drains, entries carried from one iteration to the next, the ring wrapping around)."""
import itertools
import json
import os

import numpy as np
import pytest

import bench
import fp_edges as fe
import goldenlib
import synth
from test_gpu_fast_index import _colliding_table

pytestmark = pytest.mark.gpu

LOCI = ["A", "B", "C", "DQB1", "DRB1"]
L4_OVER = {"loci_map": {"A": 1, "B": 2, "C": 3, "DRB1": 4},
           "Plan_B_Matrix": [[[1, 2, 3, 4]], [[1, 2], [3, 4]], [[1], [2], [3], [4]]]}


def _conf(d, hpf, over=None):
    open(os.path.join(d, "hpf.csv"), "w").write(hpf)
    open(os.path.join(d, "cnt.txt"), "w").write("CAU,1000.0,1.0\n")
    conf = json.load(open(os.path.join(goldenlib.GOLD, "data", "base_conf.json")))
    conf.update({"freq_file": os.path.join(d, "hpf.csv"), "pops_count_file": os.path.join(d, "cnt.txt"),
                 "freq_trim_threshold": 1e-30})
    conf.update(over or {})
    return conf


def _gpu(conf, lines, monkeypatch, probe):
    """The split fast path with GRIMB_FAST_PROBE=probe -> (six files, pair evaluations, probe kernel of the
    last launch (grimb_engine_kernel_ms 6), subjects handed on to the general kernel (3))."""
    from grim.imputation.impute import Imputation
    from grim.imputation.networkx_graph import Graph
    from grim.run_impute_def import load_config
    monkeypatch.setenv("GRIMB_HOST_EVENTS", "1")
    monkeypatch.setenv("GRIMB_KEY_WORDS", "1")
    monkeypatch.setenv("GRIMB_FAST_PROBE", probe)   # read at engine creation
    cfg = load_config(conf)
    g = Graph(cfg).build_graph()
    try:
        imp = Imputation(g, cfg)
        out = imp.impute_text("".join(lines).encode("utf8"))
        eng = g.engine(imp.workspaces[0])
        assert g.lib.grimb_engine_kernel_ms(eng, 4) >= 0, "the split fast path did not run"
        return ({k: v.decode("utf8") for k, v in out.items()}, imp.stats["pair_evals"],
                int(g.lib.grimb_engine_kernel_ms(eng, 6)), int(g.lib.grimb_engine_kernel_ms(eng, 3)))
    finally:
        monkeypatch.delenv("GRIMB_FAST_PROBE")
        g.close()


def _arms(conf, lines, monkeypatch, env=None, packed=True):
    """Both probe kernels -> [(files, evals), ...], after checking the kernel each ran and that both handed
    the same number of subjects to the general kernel; returns that number too."""
    for k, v in (env or {}).items():
        monkeypatch.setenv(k, v)
    got, handed = [], []
    for probe, kernel in (("1", 1 if packed else 0), ("2", 2 if packed else 0)):
        files, evals, ran, h = _gpu(conf, lines, monkeypatch, probe)
        assert ran == kernel, "GRIMB_FAST_PROBE=%s: probe kernel %d ran, expected %d" % (probe, ran, kernel)
        got.append((files, evals))
        handed.append(h)
    assert handed[0] == handed[1], "subjects handed to the general kernel: %r" % handed
    return got, handed[0]


def _both(conf, lines, monkeypatch, env=None, packed=True):
    """Both probe kernels and the oracle: six files and pair evaluations identical."""
    got, handed = _arms(conf, lines, monkeypatch, env, packed)
    want = fe.oracle_run(conf, lines)[:2]
    for g in got:
        fe.assert_same(g, want)
    return handed


def _name(l, a):
    return "%s*%02d:01" % (l, a + 1)


def _hpf(haps, loci=LOCI, seed=0):
    rng = np.random.RandomState(seed)
    f = rng.lognormal(0.0, 1.0, size=len(haps))
    f /= f.sum()
    return "hap,pop,freq\n" + "".join("%s,CAU,%r\n" % ("~".join(_name(l, a) for l, a in zip(loci, h)), float(x))
                                      for h, x in zip(haps, f))


def _line(tag, h1, h2, loci=LOCI):
    return "%s,%s,CAU,CAU\n" % (tag, "^".join("%s+%s" % (_name(l, a), _name(l, b)) for l, a, b in zip(loci, h1, h2)))


def test_bench_shaped_batch(tmp_path, monkeypatch):
    names, fa, ff = bench.make_table(20000)
    rows = ["hap,pop,freq\n"] + ["%s,CAU,%r\n" % ("~".join(names[l][a - 1] for l, a in enumerate(h)), float(x))
                                 for h, x in zip(fa, ff[:, 0])]
    conf = _conf(str(tmp_path), "".join(rows))
    _b, alleles = bench.make_subjects(fa, ff, 4001, bench.SUBJECT_SEED)   # not a multiple of 4
    _both(conf, bench.subject_lines(names, alleles, 0, 4001), monkeypatch)


def test_colliding_sectors(tmp_path, monkeypatch):
    names, pick, _shift, hpf = _colliding_table()
    conf = _conf(str(tmp_path), hpf)
    rng = np.random.RandomState(21)
    lines = []
    for s in range(1501):
        if s % 2 == 0:
            h1, h2 = (pick[i] for i in rng.randint(0, len(pick), size=2))
        else:
            h1, h2 = rng.randint(0, 3, size=5), rng.randint(0, 3, size=5)
        lines.append("Q%d,%s,CAU,CAU\n" % (s, "^".join("%s+%s" % (names[l][h1[l]], names[l][h2[l]]) for l in range(5))))
    _both(conf, lines, monkeypatch, {"GRIMB_FAST_INDEX_MULT": "2"})


def test_many_first_hits_no_candidate(tmp_path, monkeypatch):
    # every haplotype with DRB1 allele 0 (side 0 of the last locus, which no phase flips) and one more: a subject
    # 0/1 at every locus hits at level 1 in all 16 phases and has one candidate; one homozygous at DQB1 hits in
    # 8 phases and has none
    haps = [h + (0,) for h in itertools.product(range(2), repeat=4)] + [(1, 1, 1, 1, 1)]
    conf = _conf(str(tmp_path), _hpf(haps))
    rng = np.random.RandomState(22)
    lines = []
    for s in range(2003):
        r = rng.rand()
        if r < 0.4:
            h1, h2 = (0, 0, 0, 0, 0), (1, 1, 1, 1, 1)
        elif r < 0.8:
            h1, h2 = (0, 0, 0, 0, 0), (1, 1, 1, 0, 1)
        else:
            h1, h2 = (haps[i] for i in rng.randint(0, len(haps), size=2))
        lines.append(_line("M%d" % s, h1, h2))
    _both(conf, lines, monkeypatch)


@pytest.mark.parametrize("n", [700, 1500])
def test_long_form_and_side_record_exhaustion(n, tmp_path, monkeypatch):
    # 700: a mix of 16, 8, 4, 2 and 1 candidate phases, 328 long-form subjects within the 700 / 16 + 1024 side
    # records.  1500: every subject has 16 candidate phases, so 383 of them find no side record left
    # (1500 / 16 + 1024 = 1117) and go to the general kernel from the level-2 drain
    haps = list(itertools.product(range(2), repeat=5))
    conf = _conf(str(tmp_path), _hpf(haps, seed=1))
    rng = np.random.RandomState(23)
    lines = []
    for s in range(n):
        het = rng.randint(1, 6) if n < 1500 else 5
        h1 = tuple(rng.randint(0, 2, size=5))
        h2 = tuple(1 - a if l < het else a for l, a in enumerate(h1))
        lines.append(_line("X%d" % s, h1, h2) if s % 7 else _line("X%d" % s, (0,) * 5, (1,) * 5))
    handed = _both(conf, lines, monkeypatch)
    if n == 1500:
        assert handed >= n - (n // 16 + 1024), "side records were not exhausted: %d subjects handed on" % handed


def test_homozygous_and_unknown_alleles(tmp_path, monkeypatch):
    hpf = synth.zipf_table(400, [4, 5, 3, 3, 4], 24)
    conf = _conf(str(tmp_path), hpf)
    tab = synth.Table(hpf)
    rng = np.random.RandomState(25)
    lines = []
    for s in range(1203):
        h1, h2 = (tab.haps[i] for i in rng.choice(len(tab.haps), size=2, p=tab.p))
        k = s % 4
        if k == 0:
            h2 = h1                                   # homozygous at every locus
        sides = [[a, b] for a, b in zip(h1, h2)]
        if k in (1, 2):   # an allele the table does not hold, on one side
            l = rng.randint(0, 5)
            sides[l][k - 1] = "%s*99:99" % LOCI[l]
        lines.append("U%d,%s,CAU,CAU\n" % (s, "^".join("%s+%s" % (a, b) for a, b in sides)))
    _both(conf, lines, monkeypatch)


def test_four_loci(tmp_path, monkeypatch):
    loci = ["A", "B", "C", "DRB1"]
    hpf = synth.zipf_table(300, [5, 6, 4, 5], 26, loci=loci)
    conf = _conf(str(tmp_path), hpf, L4_OVER)
    tab = synth.Table(hpf, loci=loci)
    _both(conf, synth.typed_subjects(tab, 1001, 27, ["CAU,CAU"]), monkeypatch)


def test_chunked_host_calls(tmp_path, monkeypatch):
    # chunks of 1024 subjects: the kernels start at s_begin = 1024, 2048, ...
    hpf = synth.zipf_table(3000, [12, 20, 10, 6, 14], 28)
    conf = _conf(str(tmp_path), hpf)
    tab = synth.Table(hpf)
    _both(conf, synth.typed_subjects(tab, 3333, 29, ["CAU,CAU"]), monkeypatch, {"GRIMB_HOST_CHUNK": "1024"})


def test_general_batch_form(tmp_path, monkeypatch):
    hpf = synth.zipf_table(2000, [10, 16, 8, 6, 12], 30)
    conf = _conf(str(tmp_path), hpf)
    tab = synth.Table(hpf)
    lines = synth.typed_subjects(tab, 1500, 31, ["CAU,CAU"])
    _both(conf, lines, monkeypatch, {"GRIMB_TEXT_PACKED": "0"}, packed=False)


def test_queue_across_iterations(tmp_path, monkeypatch):
    # 120,000 subjects: with 4 CTAs of 8 warps per SM a warp takes 4 subjects per iteration and strides over
    # the batch several times.  40 % of the subjects hit at level 1 in all 16 phases, 30 % in 8, the rest in a
    # few: the queue holds entries across iterations, drains overlap the level-1 loads, the extra drain at
    # >= 64 entries runs and the ring index wraps many times.  Compared kernel against kernel (no oracle)
    haps = [h + (0,) for h in itertools.product(range(2), repeat=4)] + [(1, 1, 1, 1, 1), (0, 1, 0, 1, 1)]
    conf = _conf(str(tmp_path), _hpf(haps, seed=2))
    rng = np.random.RandomState(32)
    r = rng.rand(120000)
    rnd = rng.randint(0, 2, size=(120000, 2, 5))
    lines = []
    for s in range(120000):
        if r[s] < 0.4:
            h1, h2 = (0, 0, 0, 0, 0), (1, 1, 1, 1, 1)
        elif r[s] < 0.7:
            h1, h2 = (0, 0, 0, 0, 0), (1, 1, 1, 0, 1)
        else:
            h1, h2 = rnd[s]
        lines.append(_line("I%d" % s, h1, h2))
    (a, b), _handed = _arms(conf, lines, monkeypatch)
    fe.assert_same(b, a)


@pytest.mark.parametrize("family", ["accept", "tiny", "ties"])
def test_fp_edge_families(family, tmp_path, monkeypatch):
    d = {"accept": lambda: fe.accept_boundaries(1e-3), "tiny": fe.tiny_pairs, "ties": fe.fast_ties}[family]()
    over = {"freq_trim_threshold": fe.TRIM_SUBNORMAL} if family == "tiny" else {}
    if family == "ties":
        over["number_of_results"] = 3
    conf = d.conf(str(tmp_path), **over)
    _both(conf, d.lines(), monkeypatch)
