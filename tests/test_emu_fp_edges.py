"""CPU check of the general kernel's FP64 decision edges (the kernel source compiled for the host, tests/emu)
against the oracle: accept boundaries, exact ties, summation order and the epsilon schedule, on the designed
tables of fp_edges.py.  Files are compared byte for byte and the pair-evaluation counts must be equal (a
decision that moves a subject to another epsilon round changes only the count).  Each test also asserts,
from the instrumented oracle's records, that its batch reached the edges it is about."""
import pytest

import fp_edges as fe

POP3 = ("AAA", "BBB", "CCC")


def _check(d, tmp_path, compensated=True, **over):
    conf = d.conf(str(tmp_path), **over)
    lines = d.lines()
    files, evals, rec = fe.oracle_run(conf, lines, compensated)
    fe.assert_same(fe.emu_run(conf, lines, compensated), (files, evals))
    return rec.summary(), files


@pytest.mark.parametrize("eps", [1e-3, 1e-1, 1e-2, 1e-6])
def test_accept_boundaries_single_population(eps, tmp_path):
    s, _ = _check(fe.accept_boundaries(eps), tmp_path, epsilon=eps)
    # about a third of all evaluations fall inside the division-free band, both ways
    assert s["in_band"] >= 100 and s["in_band"] >= 0.2 * s["evals"], s
    assert s["band_accept"] >= 50 and s["band_reject"] >= 50, s
    assert s["at_eq"] >= 20 and s["same_band"] >= 10, s
    assert s["orient"] >= 10, s     # evaluations that f1 / f2 swapped would decide the other way


def test_accept_boundaries_three_populations(tmp_path):
    d = fe.Design(POP3, [600.0, 300.0, 100.0])
    s, _ = _check(fe.accept_boundaries(1e-3, d=d), tmp_path)
    assert s["f2_eq"] >= 20, s      # f2 == eps / f1 exactly: the prefix-minimum `break` test at equality
    assert s["m_ne_1_band"] >= 100 and s["band_accept"] >= 50 and s["band_reject"] >= 50, s
    assert s["at_eq"] >= 20 and s["orient"] >= 10, s


def test_tiny_and_subnormal_frequencies(tmp_path):
    s, _ = _check(fe.tiny_pairs(), tmp_path, freq_trim_threshold=fe.TRIM_SUBNORMAL)
    assert s["tiny"] >= 50 and s["tiny_accept"] >= 5, s
    assert s["plans"]["b"] >= 1, s      # the trimmed subnormal frequency sends its subjects to Plan B


@pytest.mark.parametrize("n", [1, 2, 3, 10])
def test_tied_phases(n, tmp_path):
    _, files = _check(fe.fast_ties(), tmp_path, number_of_results=n)
    if n >= 3:
        assert fe.tied_rows(files, ("pmug",)) >= 30


@pytest.mark.parametrize("k,npop", [(1, 1), (2, 2), (3, 100)])
def test_tied_populations(k, npop, tmp_path):
    _, files = _check(fe.typed_ties(), tmp_path, max_haplotypes_number_in_phase=k, number_of_pop_results=npop)
    if npop >= 2:     # with one row per subject the cut itself is what is compared
        assert fe.tied_rows(files, ("pmug", "umug_pops", "pmug_pops")) >= 5


@pytest.mark.parametrize("k", [2, 3, 5])
def test_top_k_cut_inside_equal_scores(k, tmp_path):
    s, _ = _check(fe.messy_ties(), tmp_path, max_haplotypes_number_in_phase=k)
    assert s["cut_ties"] >= 20 and s["plans"]["b"] >= 5, s


def test_save_space_mode_with_equal_sums(tmp_path):
    s, _ = _check(fe.messy_ties(), tmp_path, save_space_mode=True)
    assert s["plans"]["b"] >= 5 and s["prune_ties"] >= 20, s     # prunes whose tenth and eleventh sums are equal


@pytest.mark.parametrize("compensated", [True, False])
def test_neumaier_visible_population_sums(compensated, tmp_path):
    s, _ = _check(fe.neumaier(), tmp_path, compensated, save_space_mode=True)
    assert s["sums_differ"] >= 100, s


@pytest.mark.parametrize("planb", [True, False])
@pytest.mark.parametrize("eps", fe.epsilon_values())
def test_epsilon_schedule(eps, planb, tmp_path):
    _check(fe.schedule_design(eps), tmp_path, epsilon=eps, planb=planb)
