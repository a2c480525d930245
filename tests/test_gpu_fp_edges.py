"""GPU: the FP64 decision edges of every kernel route against the oracle, on the designed tables of
fp_edges.py -- accept boundaries within a few ulps (the division-free band of the warp kernels, the tiny
branch, the homozygous test, m != 1), exact ties, summation order (K0 marginal sums) and the epsilon
schedule (the 1e-9 cut, 40 and 41 rounds).  Each family runs through every route that serves its shape:
the split fast path (P = 1, 64-bit keys) and its fused one-kernel form, k_impute_typed (P = 3, 64- and 128-bit keys) and k_impute alone.
Files are compared byte for byte and the pair-evaluation counts must be equal."""
import numpy as np
import pytest

import fp_edges as fe
import grim_oracle as go

pytestmark = pytest.mark.gpu

POP3 = ("AAA", "BBB", "CCC")
_ref = {}


def _check(name, d, route, tmp_path, monkeypatch, **over):
    conf = d.conf(str(tmp_path), **over)
    lines = d.lines()
    if name not in _ref:
        _ref[name] = fe.oracle_run(conf, lines)
    files, evals, rec = _ref[name]
    fe.assert_same(fe.gpu_run(conf, lines, route, monkeypatch), (files, evals))
    return rec.summary(), files


@pytest.mark.parametrize("route", ["fast", "fused", "general"])
@pytest.mark.parametrize("eps", [1e-3, 1e-1, 1e-2, 1e-6])
def test_accept_boundaries_single_population(eps, route, tmp_path, monkeypatch):
    s, _ = _check("a1-%r" % eps, fe.accept_boundaries(eps), route, tmp_path, monkeypatch, epsilon=eps)
    assert s["in_band"] >= 100 and s["band_accept"] >= 50 and s["band_reject"] >= 50, s
    assert s["at_eq"] >= 20 and s["same_band"] >= 10 and s["orient"] >= 10, s


@pytest.mark.parametrize("route", ["typed1", "typed2", "general"])
def test_accept_boundaries_three_populations(route, tmp_path, monkeypatch):
    d = fe.Design(POP3, [600.0, 300.0, 100.0])
    s, _ = _check("a3", fe.accept_boundaries(1e-3, d=d), route, tmp_path, monkeypatch)
    assert s["f2_eq"] >= 20, s      # f2 == eps / f1 exactly: the prefix-minimum `break` test at equality
    assert s["m_ne_1_band"] >= 100 and s["at_eq"] >= 20 and s["orient"] >= 10, s


@pytest.mark.parametrize("route", ["fast", "fused", "general"])
def test_tiny_and_subnormal_frequencies(route, tmp_path, monkeypatch):
    s, _ = _check("tiny", fe.tiny_pairs(), route, tmp_path, monkeypatch, freq_trim_threshold=fe.TRIM_SUBNORMAL)
    assert s["tiny"] >= 50 and s["tiny_accept"] >= 5 and s["plans"]["b"] >= 1, s


@pytest.mark.parametrize("route", ["fast", "fused", "general"])
@pytest.mark.parametrize("n", [1, 2, 3, 10])
def test_tied_phases(n, route, tmp_path, monkeypatch):
    _, files = _check("ties-%d" % n, fe.fast_ties(), route, tmp_path, monkeypatch, number_of_results=n)
    if n >= 3:
        assert fe.tied_rows(files, ("pmug",)) >= 30


@pytest.mark.parametrize("route", ["typed1", "typed2", "general"])
@pytest.mark.parametrize("k,npop", [(1, 1), (2, 2), (3, 100)])
def test_tied_populations(k, npop, route, tmp_path, monkeypatch):
    _, files = _check("tpop-%d-%d" % (k, npop), fe.typed_ties(), route, tmp_path, monkeypatch,
                      max_haplotypes_number_in_phase=k, number_of_pop_results=npop)
    if npop >= 2:     # with one row per subject the cut itself is what is compared
        assert fe.tied_rows(files, ("pmug", "umug_pops", "pmug_pops")) >= 5


@pytest.mark.parametrize("k", [2, 3])
def test_top_k_cut_inside_equal_scores(k, tmp_path, monkeypatch):
    s, _ = _check("messy-%d" % k, fe.messy_ties(), "general", tmp_path, monkeypatch, max_haplotypes_number_in_phase=k)
    assert s["cut_ties"] >= 20, s


def test_save_space_mode_with_equal_sums(tmp_path, monkeypatch):
    s, _ = _check("messy-ss", fe.messy_ties(), "general", tmp_path, monkeypatch, save_space_mode=True)
    assert s["plans"]["b"] >= 5 and s["prune_ties"] >= 20, s     # prunes whose tenth and eleventh sums are equal


@pytest.mark.parametrize("planb", [True, False])
@pytest.mark.parametrize("eps", fe.epsilon_values())
def test_epsilon_schedule(eps, planb, tmp_path, monkeypatch):
    for route, pops in (("fast", ("CAU",)), ("fused", ("CAU",)), ("typed1", POP3), ("general", ("CAU",))):
        _check("sched-%r-%s-%d" % (eps, planb, len(pops)), fe.schedule_design(eps, pops), route, tmp_path, monkeypatch,
               epsilon=eps, planb=planb)


def _order_dependent_table(P):
    """Full haplotypes whose marginal sums depend on hpf row order: 0.5, 2^-54, 2^-54 summed left to right
    is 0.5, in another order 0.5 + 2^-53."""
    d = fe.Design(POP3[:P] if P > 1 else ("CAU",))
    orders = [(0.5, 2.0 ** -54, 2.0 ** -54), (2.0 ** -54, 2.0 ** -54, 0.5), (2.0 ** -54, 0.5, 2.0 ** -54),
              (0.1, 0.2, 0.3), (0.3, 0.2, 0.1)]
    for i, vals in enumerate(orders * 4):
        s = d.subject(het=[0, 1], race=None if P == 1 else ",")
        for k, (a, b) in enumerate([(0, 1), (2, 3), (1, 2)]):
            # three full haplotypes sharing A-B-C-DQB1, differing at DRB1 -> marginal sums of three rows
            h = s.hap(k)
            al = h.split("~")
            al[4] = "DRB1*%d:%02d" % (100 + s.s, 10 + k)
            for j, p in enumerate(d.pops):
                d.rows.append(("~".join(al), p, vals[(k + j + i) % 3]))
    return d


@pytest.mark.parametrize("P,kw", [(1, 1), (1, 2), (3, 1), (3, 2)])
def test_k0_marginal_sums_in_hpf_order(P, kw, tmp_path, monkeypatch):
    from emu_backend import arrays_from_oracle
    from grim.imputation.networkx_graph import Graph
    from grim.run_impute_def import load_config
    d = _order_dependent_table(P)
    conf = d.conf(str(tmp_path))
    og = go.graph_from_config(conf)
    monkeypatch.setenv("GRIMB_KEY_WORDS", str(kw))
    g = Graph(load_config(conf)).build_graph()
    monkeypatch.delenv("GRIMB_KEY_WORDS")     # arrays_from_oracle lays out 64-bit keys; the sums do not depend on it
    try:
        assert g.kw == kw
        want = arrays_from_oracle(og, g.loci)
        got = g.export()
        if kw == 1:
            assert np.array_equal(got["node_key"], want["node_key"])
        assert np.array_equal(got["node_freq"].view(np.uint64), want["freq"].view(np.uint64))
        # the table does make the sums order-dependent
        f = want["freq"][og.n_full:]
        assert np.any(f == 0.5) and np.any(f == 0.5 + 2.0 ** -53)
    finally:
        g.close()
