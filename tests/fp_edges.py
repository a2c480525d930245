"""Tables and subjects built to sit on the FP64 decision edges of the imputation, an instrumented oracle
that shows which edges a batch reached, and runners for the three kernel routes and the emulation build.

Every decision the kernels take must be bit-exact for the output files to match the reference byte for
byte: the accept test of a candidate pair (eps / f1 against f2 and m * f2), the epsilon round a subject
accepts in, the rank of tied rows, which tied entries a top-K cap or save_space_mode keeps, and the order
of every sum.  Frequencies drawn from a distribution never come within a few ulps of a threshold, are
never exactly equal and rarely make a sum depend on its order, so the families here are built from
chosen doubles instead:

- every designed subject has alleles of its own (locus name, subject number, variant), so the
  frequencies of one subject are tuned without touching any other;
- hpf rows are written with %r, which round-trips every double;
- the builders do not assume which haplotype of a phase the oracle takes as f1: they put the product
  f1 * f2 * m on the threshold, and the records of the instrumented oracle say what was reached.
"""
import builtins
import contextlib
import itertools
import json
import math
import os

import numpy as np

import goldenlib
import grim_oracle as go

LOCI = ["A", "B", "C", "DQB1", "DRB1"]
BAND = 2.0 ** -50        # half-width of the division-free accept band of the warp kernels (FastPair)
TINY = 1.0e-280          # below this bound the warp kernels always divide


def ulp_step(x, d):
    """x moved by d ulps (d may be negative)."""
    for _ in range(abs(d)):
        x = math.nextafter(x, math.inf if d > 0 else -math.inf)
    return x


def chain(eps0):
    """The epsilon rounds of the reference (impute.py:1665-1673): /= 10, cut to 0 below 1e-9."""
    out = []
    e = eps0
    while e > 0:
        e /= 10
        if e < 1.0e-9:
            e = 0.0
        out.append(e)
    return out


def smallest_eps_with_rounds(n):
    """The smallest positive double whose epsilon chain has exactly n rounds (n >= 2)."""
    lo, hi = 1e-300, 1e300
    assert len(chain(lo)) <= n <= len(chain(hi))
    # the number of rounds is non-decreasing in eps: bisect on the bit patterns
    a, b = int(np.float64(lo).view(np.int64)), int(np.float64(hi).view(np.int64))
    while b - a > 1:
        c = (a + b) // 2
        if len(chain(float(np.int64(c).view(np.float64)))) >= n:
            b = c
        else:
            a = c
    e = float(np.int64(b).view(np.float64))
    assert len(chain(e)) == n and len(chain(math.nextafter(e, 0.0))) == n - 1
    return e


# --------------------------------------------------------------------------- builders
class Subject(object):
    """One designed subject: heterozygous at the loci `het` (indices into LOCI), its own alleles.
    A haplotype is named by a bit mask over the loci: bit l set = the second allele of locus l."""

    def __init__(self, design, s, het, race):
        self.d, self.s, self.het, self.race = design, s, sorted(het), race
        self.hmask = sum(1 << l for l in self.het)

    def allele(self, l, v):
        return "%s*%d:%02d" % (LOCI[l], 100 + self.s, v + 1)

    def hap(self, mask):
        return "~".join(self.allele(l, (mask >> l) & 1) for l in range(len(LOCI)))

    def phase_pairs(self):
        """(mask, complement) of every phase: the masks whose highest heterozygous bit is clear."""
        if not self.het:
            return [(0, 0)]
        top = 1 << self.het[-1]
        out = []
        for k in range(1 << len(self.het)):
            m = sum(1 << l for i, l in enumerate(self.het) if (k >> i) & 1)
            if not m & top:
                out.append((m, m ^ self.hmask))
        return out

    def set(self, mask, freq):
        """freq: one double (first population) or {population: double}."""
        if not isinstance(freq, dict):
            freq = {self.d.pops[0]: freq}
        for p, f in freq.items():
            self.d.rows.append((self.hap(mask), p, float(f)))

    def pair(self, k, f_a, f_b):
        """Frequencies of the two haplotypes of phase k (order of phase_pairs)."""
        a, b = self.phase_pairs()[k]
        self.set(a, f_a)
        if b != a:
            self.set(b, f_b)

    def line(self):
        gl = "^".join("%s+%s" % (self.allele(l, 0), self.allele(l, 1 if l in self.het else 0)) for l in range(len(LOCI)))
        return "E%d,%s%s\n" % (self.s, gl, "," + self.race if self.race is not None else "")


class Design(object):
    """A table and a subject list built together."""

    def __init__(self, pops=("CAU",), counts=None):
        self.pops = list(pops)
        self.counts = counts or [1000.0] * len(self.pops)
        self.rows = []
        self.subjects = []
        self.extra_lines = []

    def subject(self, het=(), race=None):
        if race is None and len(self.pops) == 1:
            race = "%s,%s" % (self.pops[0], self.pops[0])
        s = Subject(self, len(self.subjects), het, race)
        self.subjects.append(s)
        return s

    def _m(self, race, p1, p2):
        """M[p1][p2] of the prior matrix the oracle builds for a race field pair (1.0 for P = 1)."""
        if len(self.pops) == 1 or not any(r in self.pops for r in race.replace(";", ",").split(",")):
            return 1.0      # no known race: M = ones (UNK_priors MR)
        base = json.load(open(os.path.join(goldenlib.GOLD, "data", "base_conf.json")))
        cfg = go.load_config({"populations": self.pops, "priority": base["priority"]})
        tot = sum(self.counts)
        o = go.OracleImputation(None, cfg, np.array([float(repr(float(c / tot))) for c in self.counts]))
        r1, r2 = race.split(",")
        M = o.prior_matrix(r1.split(";"), r2.split(";"))
        return float(M[self.pops.index(p1)][self.pops.index(p2)])

    def hpf(self):
        return "hap,pop,freq\n" + "".join("%s,%s,%r\n" % r for r in self.rows)

    def counts_text(self):
        tot = sum(self.counts)
        return "".join("%s,%r,%r\n" % (p, float(c), float(c / tot)) for p, c in zip(self.pops, self.counts))

    def lines(self):
        return [s.line() for s in self.subjects] + list(self.extra_lines)

    def conf(self, d, **over):
        """Writes the table into directory d -> a run_impute_def-style configuration."""
        with open(os.path.join(d, "hpf.csv"), "w") as f:
            f.write(self.hpf())
        with open(os.path.join(d, "cnt.txt"), "w") as f:
            f.write(self.counts_text())
        conf = json.load(open(os.path.join(goldenlib.GOLD, "data", "base_conf.json")))
        conf.update({"populations": self.pops, "freq_file": os.path.join(d, "hpf.csv"),
                     "pops_count_file": os.path.join(d, "cnt.txt"), "freq_trim_threshold": 1e-300,
                     "UNK_priors": "MR"})
        conf.update(over)
        return conf


# --------------------------------------------------------------------------- instrumented oracle
class Eval(object):
    __slots__ = ("eps", "f1", "f2", "m", "same", "accepted", "in_band", "tiny", "at_eq", "orient")

    def __init__(self, eps, f1, f2, m, same, accepted):
        self.eps, self.f1, self.f2, self.m, self.same, self.accepted = eps, f1, f2, m, same, accepted
        t = min(f2, m * f2 * 0.5 if same else m * f2)
        b = f1 * t
        self.tiny = not b > TINY
        self.in_band = (not self.tiny) and b * (1 - BAND) < eps < b * (1 + BAND)
        x = eps / f1
        self.at_eq = accepted and (f2 == x or m * f2 == (x * 2 if same else x))
        # the decision with the two haplotypes swapped (eps / f2 against f1) differs
        self.orient = _accept(eps, f2, f1, m, same) != accepted


def _accept(eps, f1, f2, m, same):
    x = eps / f1
    return f2 >= x and m > 0 and m * f2 >= (x * 2 if same else x)


class Records(object):
    def __init__(self):
        self.evals = []
        self.plans = {}          # subject id -> plan letter of its last evaluation ("a", "b", "c")
        self.prune_ties = 0      # save_space prunes whose 10th and 11th largest sums are equal
        self.prunes = 0
        self.sums_differ = 0     # float sums where Neumaier compensation changes the result
        self.float_sums = 0
        self.cut_ties = 0        # max_haplotypes_number_in_phase cuts between two equal weights

    def summary(self):
        e = self.evals
        return {"evals": len(e), "in_band": sum(r.in_band for r in e),
                "band_accept": sum(r.in_band and r.accepted for r in e),
                "band_reject": sum(r.in_band and not r.accepted for r in e),
                "at_eq": sum(r.at_eq for r in e), "f2_eq": sum(r.f2 == r.eps / r.f1 for r in e), "tiny": sum(r.tiny for r in e),
                "tiny_accept": sum(r.tiny and r.accepted for r in e),
                "orient": sum(r.orient for r in e), "same_band": sum(r.same and r.in_band for r in e),
                "m_ne_1_band": sum(r.m != 1.0 and r.in_band for r in e),
                "plans": {p: list(self.plans.values()).count(p) for p in "abc"},
                "prunes": self.prunes, "prune_ties": self.prune_ties,
                "float_sums": self.float_sums, "sums_differ": self.sums_differ, "cut_ties": self.cut_ties}


def _fold(v):
    v = list(v)
    if not v:
        return 0
    f = 0 + v[0]
    for x in v[1:]:
        f = f + x
    return f


@contextlib.contextmanager
def instrumented(rec, compensated=True):
    """Wraps the oracle's pair loop, save_space prune, subject entry and sum() (plain left fold when
    compensated is False: the summation of CPython before 3.12)."""
    O = go.OracleImputation
    o_pairs, o_combine, o_one, o_flatten = O._pairs, O._combine, O.impute_one, O._flatten

    def flatten(self, probs):
        w = sorted((v[j] * self.M[j][j] for v in probs for j in range(len(v)) if v[j] > 0), reverse=True)
        rec.cut_ties += len(w) > self.top_k and w[self.top_k - 1] == w[self.top_k]
        return o_flatten(self, probs)

    def pairs(self, haps1, haps2, top1, top2, eps, acc, muug):
        before, n = self.pair_evals, 0
        for _w1, f1, k1, p1 in top1:
            x = eps / f1
            for _w2, f2, k2, p2 in top2:
                n += 1
                m = float(self.M[p1][p2])
                same = haps1[k1] == haps2[k2]
                rec.evals.append(Eval(eps, f1, f2, m, same, _accept(eps, f1, f2, m, same)))
                if not f2 >= x:
                    break
        o_pairs(self, haps1, haps2, top1, top2, eps, acc, muug)
        assert self.pair_evals - before == n, "the instrumented copy of the pair loop drifted from the oracle"

    def combine(self, new, acc, planc=False):
        if self.save_space:
            for d in (acc, new):
                if len(d) > 10:
                    rec.prunes += 1
                    s = sorted((go.sum(v) for v in d.values()), reverse=True)
                    rec.prune_ties += s[9] == s[10]
        return o_combine(self, new, acc, planc)

    def one(self, gl, race1, race2):
        out = o_one(self, gl, race1, race2)
        rec.plans[gl] = self.plan
        return out

    def summ(v, start=0):
        v = list(v)
        if any(isinstance(x, float) for x in v):
            rec.float_sums += 1
            c = builtins.sum(v, start)
            f = _fold([start] + v) if start else _fold(v)
            rec.sums_differ += c != f
            return c if compensated else f
        return builtins.sum(v, start)

    O._pairs, O._combine, O.impute_one, O._flatten = pairs, combine, one, flatten
    go.sum = summ
    try:
        yield rec
    finally:
        O._pairs, O._combine, O.impute_one, O._flatten = o_pairs, o_combine, o_one, o_flatten
        del go.sum


def oracle_run(conf, lines, compensated=True):
    """-> (six file texts, pair evaluations, Records)."""
    rec = Records()
    with instrumented(rec, compensated):
        g = go.graph_from_config(conf)
        cfg = go.load_config(conf)
        o = go.OracleImputation(g, cfg, go.count_by_prob_from_file(len(cfg["pops"]), conf["pops_count_file"]))
        files = o.impute_lines(lines)
    return files, o.pair_evals, rec


# --------------------------------------------------------------------------- product runs
def emu_run(conf, lines, compensated=True):
    """The kernel source compiled for the host (tests/emu): the general kernel's per-subject algorithm."""
    from emu_backend import EmuGraph, emu_imputation
    from grim.run_impute_def import load_config
    eg = EmuGraph(go.graph_from_config(conf), conf["loci_map"])
    imp = emu_imputation(eg, load_config(conf))
    imp.cfg.compensated_sum = 1 if compensated else 0
    files = imp.impute_lines(lines)
    return {k: "".join(v) for k, v in files.items()}, imp.stats["pair_evals"]


def gpu_run(conf, lines, route, monkeypatch, compensated=True):
    """One of the kernel routes on the GPU, through the C++ text pipeline:
    fast     k_fast_probe + k_fast_score (P = 1, 64-bit keys)
    fused    k_impute_fast, the one-kernel form of the same path (GRIMB_FAST_SPLIT=0)
    typed1/2 k_impute_typed with 64- / 128-bit keys (P > 1)
    general  k_impute alone (GRIMB_FAST=0: no warp-per-subject kernel)
    Asserts that the route was taken; -> (six file texts, pair evaluations)."""
    from grim.imputation.impute import Imputation
    from grim.imputation.networkx_graph import Graph
    from grim.run_impute_def import load_config
    monkeypatch.setenv("GRIMB_HOST_EVENTS", "1")    # kernel timing events (read at engine creation)
    monkeypatch.setenv("GRIMB_KEY_WORDS", "2" if route == "typed2" else "1")
    monkeypatch.setenv("GRIMB_FAST", "0" if route == "general" else "1")
    monkeypatch.setenv("GRIMB_FAST_SPLIT", "0" if route == "fused" else "1")
    cfg = load_config(conf)
    g = Graph(cfg).build_graph()
    try:
        imp = Imputation(g, cfg)
        imp.cfg.compensated_sum = 1 if compensated else 0
        out = imp.impute_text("".join(lines).encode("utf8"))
        eng = g.engine(imp.workspaces[0])
        ms = [g.lib.grimb_engine_kernel_ms(eng, w) for w in range(5)]
        if route == "fast":
            assert ms[4] >= 0, "the split fast path did not run"
        elif route == "fused":
            assert ms[0] >= 0 and ms[4] < 0, "k_impute_fast did not run"
        elif route.startswith("typed"):
            assert ms[2] >= 0, "k_impute_typed did not run"
            assert g.kw == (2 if route == "typed2" else 1)
        else:
            assert ms[0] < 0 and ms[2] < 0 and ms[4] < 0, "a warp-per-subject kernel ran"
            assert ms[1] >= 0, "k_impute did not run"
        return {k: v.decode("utf8") for k, v in out.items()}, imp.stats["pair_evals"]
    finally:
        monkeypatch.delenv("GRIMB_KEY_WORDS")
        monkeypatch.delenv("GRIMB_FAST")
        monkeypatch.delenv("GRIMB_FAST_SPLIT")
        g.close()


def assert_same(got, want):
    files, evals = got
    rfiles, revals = want
    for k in goldenlib.KEYS:
        assert files[k] == rfiles[k], "%s differs" % k
    assert evals == revals, "pair evaluations: %d, oracle %d" % (evals, revals)


# --------------------------------------------------------------------------- families
F1S = (0.3, 0.07, 1.0 / 3.0, 0.0123456789)      # first frequencies of the boundary pairs


def accept_boundaries(eps0, pops=("CAU",), d=None):
    """Family A.  Subjects whose accept decision sits within a few ulps of a threshold:
    - one candidate phase, f1 * f2 on every positive round of the chain of eps0, d in -2..2 ulps
      (moves the round it accepts in: only the pair-evaluation count shows it);
    - two candidate phases: (0.3, 0.2) accepts in the first round, (f3, f4) sits on the final
      threshold MaxProb / 100000 (decides whether it is a PMUG row);
    - homozygous subjects, f * f on 2 * eps (the `same` test);
    - long form: four and five heterozygous loci (8 and 16 candidate phases), every phase but the
      first on the final threshold;
    - with P > 1: the two haplotypes in different populations, so m = M[p1][p2] != 1."""
    d = d or Design(pops)
    P = len(d.pops)
    races = ["%s,%s" % (d.pops[0], d.pops[0])] if P == 1 else ["%s,%s" % (d.pops[0], d.pops[1]), "%s,%s" % (d.pops[2], d.pops[0]), ","]
    rounds = [e for e in chain(eps0) if e > 0]

    def pop_pair(s, race):
        if P == 1:
            return d.pops[0], d.pops[0], 1.0
        r1, r2 = race.split(",")
        return r1 or d.pops[1], r2 or d.pops[1], None

    def put(s, k, fa, fb, p1, p2):
        s.pair(k, {p1: fa}, {p2: fb})

    for ri, e in enumerate(rounds):
        for fi, f1 in enumerate(F1S):
            race = races[(ri + fi) % len(races)]
            for dd in range(-2, 3):
                s = d.subject(het=[0], race=race)
                p1, p2, _ = pop_pair(s, race)
                m = d._m(race, p1, p2)
                x = e / f1
                put(s, 0, f1, ulp_step(x / m if m != 1.0 else x, dd), p1, p2)
        # homozygous: f * f = 2 * eps
        for dd in range(-3, 4):
            s = d.subject(het=[], race=races[ri % len(races)])
            p1 = d.pops[0]
            m = d._m(s.race, p1, p1)
            s.set(0, {p1: ulp_step(math.sqrt(2 * e / m), dd)})
    # two candidates on the final threshold, and the long form
    for het in ([0, 1], [0, 1, 2, 3], [0, 1, 2, 3, 4]):
        for f3 in (0.001, 0.0007, 1.0 / 7.0):
            for dd in range(-2, 3):
                race = races[dd % len(races)]
                s = d.subject(het=het, race=race)
                p1, p2, _ = pop_pair(s, race)
                m = d._m(race, p1, p2)
                s.pair(0, {p1: 0.3}, {p2: 0.2})
                mx = 0.3 * 0.2 * m * 2
                fin = mx / 100000
                for k in range(1, len(s.phase_pairs())):
                    f = f3 * (1 + k / 64.0)
                    s.pair(k, {p1: f}, {p2: ulp_step(fin / f / m if m != 1.0 else fin / f, dd + (k % 3) - 1)})
    return d




def tiny_pairs(d=None):
    """Family A, the branch that always divides: f1 * f2 <= 1e-280, subnormal frequencies, and subnormal
    frequencies on both sides of a subnormal trim threshold (freq_trim_threshold / count)."""
    d = d or Design()
    vals = [(1e-150, 1e-140), (2.0 ** -1000, 2.0 ** -20), (5e-320, 0.5), (1e-310, 1e-5), (2e-312, 0.25),
            (5e-313, 0.25), (1e-300, 1e-300), (3e-308, 2e-308)]
    for fa, fb in vals:
        s = d.subject(het=[0])
        s.pair(0, fa, fb)
        # with a second, ordinary phase: the tiny one must stay out at MaxProb / 100000
        s = d.subject(het=[0, 1])
        s.pair(0, 0.3, 0.2)
        s.pair(1, fa, fb)
    s = d.subject(het=[])     # homozygous, subnormal
    s.set(0, 4e-320)
    return d


TRIM_SUBNORMAL = 1e-309       # / count 1000 -> 1e-312: 5e-313 is trimmed, 2e-312 is kept


def fast_ties(d=None):
    """Family B, P = 1: phases with exactly equal probabilities (dyadic frequencies) and probabilities
    one ulp apart, in every assignment to the phases, so a result limit cuts inside the tie."""
    d = d or Design()
    up = 2.0 ** -3 * (1 + 2.0 ** -52)
    dn = 2.0 ** -3 * (1 - 2.0 ** -53)
    vals = [(2.0 ** -2, 2.0 ** -4), (2.0 ** -3, 2.0 ** -3), (2.0 ** -1, 2.0 ** -5), (up, 2.0 ** -3)]
    for perm in itertools.permutations(range(4)):
        s = d.subject(het=[0, 1, 2])
        for k, j in enumerate(perm):
            s.pair(k, *vals[j])
    for perm in itertools.permutations(range(3)):
        s = d.subject(het=[1, 3, 4])
        v = [vals[1], (dn, 2.0 ** -3), vals[0]]
        for k, j in enumerate(perm):
            s.pair(k, *v[j])
        s.pair(3, 2.0 ** -2, 2.0 ** -4)
    for het in ([0, 1, 2, 3], [0, 1, 2, 3, 4]):      # long form: 8 and 16 tied candidates
        for variant in range(4):
            s = d.subject(het=het)
            for k in range(len(s.phase_pairs())):
                fa = 2.0 ** -5
                if variant == 1 and k % 3 == 1:
                    fa = up
                if variant == 2 and k % 4 == 2:
                    fa = dn
                if variant == 3:
                    fa = 2.0 ** -(2 + k % 3)
                    s.pair(k, fa, 2.0 ** -10 / fa)
                    continue
                s.pair(k, fa, 2.0 ** -5)
    return d


def typed_ties(d=None):
    """Family B, P = 3: haplotypes with equal frequencies in every population (equal counts, so w = f * M[j][j]
    ties across populations when the diagonal is equal) and population-pair sums that tie."""
    d = d or Design(("AAA", "BBB", "CCC"))
    races = [",", "AAA,BBB", "CCC,CCC", "AAA;BBB,CCC"]
    for r in range(len(races)):
        for het in ([0], [0, 1], [2, 4], []):
            s = d.subject(het=het, race=races[r])
            for k, (a, b) in enumerate(s.phase_pairs()):
                fa = 2.0 ** -(3 + k)
                s.set(a, {p: fa for p in d.pops})
                if b != a:
                    s.set(b, {p: 2.0 ** -4 for p in d.pops[: 2 + (k + r) % 2]})
    return d


def messy_ties(d=None, seed=5):
    """Family B, general kernel: ambiguous subjects (two or three alleles per locus side) whose candidate
    haplotypes have equal frequencies, so a small max_haplotypes_number_in_phase cuts inside a run of
    equal scores; and Plan B subjects whose blocks have more than ten equal marginal sums (save_space_mode
    cuts at the tenth place).  Frequencies are dyadic, and P = 3 with equal counts."""
    rng = np.random.RandomState(seed)
    d = d or Design(("AAA", "BBB", "CCC"))
    n0 = len(d.subjects)
    for i in range(60):
        s = d.subject(race=",")
        amb = 2 + i % 2
        sides = [[[s.allele(l, v) for v in range(amb)], [s.allele(l, amb + v) for v in range(amb)]] for l in range(5)]
        all_al = [sides[l][0] + sides[l][1] for l in range(5)]
        if i % 3 == 2:
            # Plan B: every A-B-C of a side list with foreign DQB1-DRB1 and every DQB1-DRB1 with foreign A-B-C, so the
            # blocks of Plan_B_Matrix row 2 have up to 27 entries, most with equal sums
            for side in ([sides[l][0] for l in range(5)], [sides[l][1] for l in range(5)]):
                for j, abc in enumerate(itertools.product(*side[:3])):
                    f = 2.0 ** -9 if j % 7 == 3 else 2.0 ** -8
                    for p in d.pops:
                        d.rows.append(("~".join(list(abc) + [s.allele(3, 20 + j), s.allele(4, 20 + j)]), p, f))
                for j, dq in enumerate(itertools.product(*side[3:])):
                    for p in d.pops:
                        d.rows.append(("~".join([s.allele(l, 40 + j) for l in range(3)] + list(dq)), p, 2.0 ** -7))
        else:
            for j in range(40):
                h = [all_al[l][rng.randint(len(all_al[l]))] for l in range(5)]
                f = [2.0 ** -6, 2.0 ** -7, 2.0 ** -6][j % 3]
                for p in d.pops[: 1 + j % 3]:
                    d.rows.append(("~".join(h), p, f))
        s.gl = "^".join("/".join(a) + "+" + "/".join(b) for a, b in sides)
    lines = ["E%d,%s,,\n" % (s.s, s.gl) for s in d.subjects[n0:]]
    d.subjects = d.subjects[:n0]
    d.extra_lines.extend(lines)
    return d


def neumaier(d=None):
    """Family C: population vectors whose Python sum() depends on compensation ([0.25, 2^-55, 2^-55]
    and the like) on subjects that reach Plan B with save_space_mode and Plan C, P = 3."""
    d = d or Design(("AAA", "BBB", "CCC"))
    vecs = [(0.25, 2.0 ** -55, 2.0 ** -55), (2.0 ** -55, 0.25, 2.0 ** -55), (1.0, 1e-16, 1e-16),
            (0.1, 0.2, 0.3), (2.0 ** -55, 2.0 ** -55, 0.25)]
    n0 = len(d.subjects)
    for i in range(12):
        s = d.subject(race=",")
        amb = 3
        sides = [[[s.allele(l, v) for v in range(amb)], [s.allele(l, amb + v) for v in range(amb)]] for l in range(5)]
        all_al = [sides[l][0] + sides[l][1] for l in range(5)]
        for j in range(26):
            h = [all_al[l][(j * (l + 1) + i) % len(all_al[l])] for l in range(5)]
            # Plan B / C: no full haplotype of the subject's own alleles; marginals with Neumaier-visible vectors
            for l in ((3, 4) if j % 2 else (0, 1, 2)):
                h[l] = s.allele(l, 20 + j % 5)
            v = vecs[(i + j) % len(vecs)]
            for p, f in zip(d.pops, v):
                d.rows.append(("~".join(h), p, f))
        if i % 4 == 3:   # an allele absent from the table: the missing-data path and Plan C
            sides[2][0][0] = "C*99:%02d" % (1 + i % 7)
        s.gl = "^".join("/".join(a) + "+" + "/".join(b) for a, b in sides)
    lines = ["E%d,%s,,\n" % (s.s, s.gl) for s in d.subjects[n0:]]
    d.subjects = d.subjects[:n0]
    d.extra_lines.extend(lines)
    return d


def epsilon_values():
    """Family D: epsilon values that put a round of the chain next to the 1e-9 cut, the smallest with
    40 and 41 rounds (the warp kernels keep at most 40), and 1e300."""
    e8 = 1e-8
    out = [e8, math.nextafter(e8, 0.0), math.nextafter(e8, 1.0), 1e-9 * 10, math.nextafter(1e-9 * 10, 1.0)]
    # a round that lands exactly on the double 1e-9 (the cut is eps < 1e-9)
    x = 1e-9 * 100
    for dd in range(-4, 5):
        y = ulp_step(x, dd)
        if chain(y)[1] == 1e-9:
            out.append(y)
            break
    out += [smallest_eps_with_rounds(40), smallest_eps_with_rounds(41), 1e300]
    return sorted(set(out))


def schedule_design(eps0, pops=("CAU",)):
    """Subjects that accept only in late rounds of the chain of eps0 (and at 0), plus the boundary subjects
    of the last positive rounds."""
    d = Design(pops)
    rounds = [e for e in chain(eps0) if e > 0]
    for e in rounds[-3:]:
        for f1 in F1S[:2]:
            for dd in range(-1, 2):
                s = d.subject(het=[0], race=None if len(pops) == 1 else "%s,%s" % (pops[0], pops[0]))
                s.pair(0, {pops[0]: f1}, {pops[0]: ulp_step(e / f1, dd)})
    for f in (1e-6, 1e-12, 1e-30):      # accept only in the round with eps = 0 (or never before the chain ends)
        s = d.subject(het=[0, 2], race=None if len(pops) == 1 else "%s,%s" % (pops[0], pops[0]))
        s.pair(0, {pops[0]: f}, {pops[0]: f})
        s.pair(1, {pops[0]: f * 0.5}, {pops[0]: f})
    s = d.subject(het=[0], race=None if len(pops) == 1 else "%s,%s" % (pops[0], pops[0]))
    s.pair(0, {pops[0]: 0.5}, {pops[0]: 0.25})
    return d


def tied_rows(files, keys=("pmug", "umug_pops", "pmug_pops")):
    """Adjacent rows of one subject with the same printed probability, in the given output files."""
    n = 0
    for k in keys:
        prev = None
        for row in files[k].splitlines():
            f = row.split(",")
            sid, p = f[0], f[-2]
            n += prev == (sid, p)
            prev = (sid, p)
    return n
