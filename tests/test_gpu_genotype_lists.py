"""GPU: the device-resident route for genotypes with allele ambiguity (Imputation.encode_genotype_lists /
impute_genotype_lists: ragged allele lists -> grimb_batch_from_genotype_lists -> the imputation kernels ->
grimb_results_rows -> ragged row tensors), with per-subject phase masks and the EM-facing modes (em_mr's
hap;pop rows through GenotypeResults.pmug_pairs, em).  The rows are rendered into the six output texts by the
renderer of test_gpu_genotype_api.py, plus the hap;pop row format of em_mr, and compared byte for byte with the
text route on the same lines (impute_text, or impute_lines for phase masks and the EM modes) -- and with the
reference's own files for every golden case whose lines all take this route."""
import ctypes as C
import json
import os

import numpy as np
import pytest

import goldenlib
import synth
from test_gpu_genotype_api import _split, render

pytestmark = pytest.mark.gpu

ST_SKIPPED = 4
E_ARG = -1          # GRIMB_E_ARG
KINDS = ("umug", "pmug", "umug_pops", "pmug_pops")


def _graph(conf, monkeypatch=None, kw=None):
    from grim.imputation.impute import Imputation
    from grim.imputation.networkx_graph import Graph
    from grim.run_impute_def import load_config
    if kw is not None:
        monkeypatch.setenv("GRIMB_KEY_WORDS", str(kw))
    cfg = load_config(conf)
    g = Graph(cfg).build_graph()
    return g, Imputation(g, cfg)


def _readme_conf():
    _t, conf, _l, _e = goldenlib.load_case("g1_readme_donor")
    return conf


def _np(x):
    """numpy view of a result array (CUDA tensors of unsigned types go through their signed twins)."""
    if x is None or not hasattr(x, "cpu"):
        return x
    import torch
    signed = {torch.uint16: (torch.int16, np.uint16), torch.uint32: (torch.int32, np.uint32)}
    if x.dtype in signed:
        return x.view(signed[x.dtype][0]).cpu().numpy().view(signed[x.dtype][1])
    return x.cpu().numpy()


def render_lists(res, imp, sids, raws, unknown, em_mr=False):
    """render() of test_gpu_genotype_api, with the .pmug rows of em_mr written as write_best_hap_race_pairs writes
    them ("sid,hap;pop,hap;pop,prob,k")."""
    out = render(res, imp, sids, raws, unknown)
    if not em_mr or not imp.config["output_haplotypes"]:
        return out
    L = imp.L
    r, p, o, pairs = _np(res.pmug).astype(np.int64), _np(res.pmug_prob), _np(res.pmug_off), _np(res.pmug_pairs)
    st, fl = _np(res.status), _np(res.flags)
    pop = lambda x: "all_pops" if x == 0xFFFF else res.populations[x]

    def name(s, l, i):
        al = res.alleles[l]
        return al[i - 1] if 1 <= i <= len(al) else unknown[s][(l, i)]
    rows = []
    for s, sid in enumerate(sids):
        if fl[s] & 4:
            continue
        for k, q in enumerate(range(o[s], o[s + 1])):
            h = ["~".join(name(s, l, int(r[q, x, l])) for l in range(L) if r[q, x, l]) for x in (0, 1)]
            rows.append("%s,%s;%s,%s;%s,%r,%d\n" % (sid, h[0], pop(int(pairs[q, 0])), h[1], pop(int(pairs[q, 1])), float(p[q]), k))
    out["pmug"] = "".join(rows)
    assert st.shape[0] == len(sids)
    return out


def _lists_run(imp, lines, cuda=True, em_mr=False, em=False):
    """Lines -> (the list route's six texts, results, the lines it took).  Lines the encoder sends to the text path
    (problem, fault, foreign loci), lines the line parser rejects and, with phase masks configured, lines whose id
    has no mask (the text path faults them) are left out."""
    import torch
    parsed = _split(lines)
    keep = [i for i, x in enumerate(parsed) if x is not None]
    counts, alleles, unknown, text_path = imp.encode_genotype_lists([parsed[i][1] for i in keep])
    drop = set(text_path)
    masks = None
    if imp.phase_masks is not None:
        masks, missing = imp.phase_masks_for([parsed[i][0] for i in keep])
        drop |= set(missing)
    ok = [j for j in range(len(keep)) if j not in drop]
    n = counts.astype(np.int64).sum((1, 2))
    off = np.concatenate([[0], np.cumsum(n)])
    alleles = np.concatenate([alleles[off[j]:off[j + 1]] for j in ok] + [np.zeros(0, np.uint16)])
    counts, unknown = counts[ok], [unknown[j] for j in ok]
    taken = [lines[keep[j]] for j in ok]
    pri = [imp.prior_index(parsed[keep[j]][2], parsed[keep[j]][3]) for j in ok]
    pm = masks[ok] if masks is not None else None
    dev = imp.netGraph.device
    if cuda:
        counts, alleles = torch.from_numpy(counts).cuda(dev), torch.from_numpy(alleles).cuda(dev)
        pm = torch.from_numpy(pm).cuda(dev) if pm is not None else None
    res = imp.impute_genotype_lists(counts, alleles, pri, phase_mask=pm, em_mr=em_mr, em=em)
    sids = [parsed[keep[j]][0] for j in ok]
    return render_lists(res, imp, sids, taken, unknown, em_mr), res, taken


def _text(imp, lines, em_mr=False, em=False, host=False):
    if host or em_mr or em or imp.phase_masks is not None:
        return {k: "".join(v) for k, v in imp.impute_lines(lines, em_mr=em_mr, em=em).items()}
    out = imp.impute_text("".join(lines).encode("utf8"))
    return {k: v.decode("utf8") for k, v in out.items()}


def _assert_files(got, want, what):
    for k in goldenlib.KEYS:
        if got[k] != want[k]:
            a, b = got[k].splitlines(), want[k].splitlines()
            i = next((j for j in range(min(len(a), len(b))) if a[j] != b[j]), min(len(a), len(b)))
            raise AssertionError("%s: %s differs at row %d: %r vs %r (%d / %d rows)" % (
                what, k, i, a[i] if i < len(a) else None, b[i] if i < len(b) else None, len(a), len(b)))


def _compare(imp, lines, what, cuda=True, em_mr=False, em=False):
    got, res, taken = _lists_run(imp, lines, cuda, em_mr, em)
    _assert_files(got, _text(imp, taken, em_mr, em), what)
    return got, res, taken


def _same(a, b, pair_evals=True):
    for k in ("status", "flags", "plan_umug", "plan_pmug", "tot_umug", "tot_pmug"):
        assert np.array_equal(_np(getattr(a, k)), _np(getattr(b, k))), k
    for k in KINDS:
        for suf in ("", "_off"):
            assert np.array_equal(_np(getattr(a, k + suf)), _np(getattr(b, k + suf))), k + suf
        assert _np(getattr(a, k + "_prob")).tobytes() == _np(getattr(b, k + "_prob")).tobytes(), k
    assert (a.pmug_pairs is None) == (b.pmug_pairs is None)
    if a.pmug_pairs is not None:
        assert np.array_equal(_np(a.pmug_pairs), _np(b.pmug_pairs))
    if pair_evals:
        assert a.pair_evals == b.pair_evals


def _no_rows(res, s):
    for k in KINDS:
        o = _np(getattr(res, k + "_off"))
        assert o[s + 1] == o[s], (s, k)


# --------------------------------------------------------------------------- every golden case
@pytest.mark.parametrize("name", goldenlib.case_names())
def test_golden_case_through_the_list_route(name):
    _t, conf, lines, exp = goldenlib.load_case(name)
    em_mr = conf.pop("_hap_pop_pair")
    if conf.get("Plan_A_Matrix"):
        conf["planb"] = False    # under a matrix the reference's Plan B is not defined (DESIGN 7)
    g, imp = _graph(conf)
    try:
        got, res, taken = _compare(imp, lines, name, em_mr=em_mr)
        if taken:
            assert g.lib.grimb_engine_kernel_ms(g.engine(imp.workspaces[0]), 9) >= 0
        assert (res.pmug_pairs is not None) == em_mr
        if conf.get("Plan_A_Matrix"):
            return
        # lines whose id has no phase mask: the text path writes them raw to .problem and nothing else
        no_mask = []
        if imp.phase_masks is not None:
            no_mask = [ln for ln in lines if _split([ln])[0] is not None and _split([ln])[0][0] not in imp.phase_masks]
        if len(taken) + len(no_mask) == len(lines) and not (no_mask and got["problem"]):
            if no_mask:
                got = dict(got, problem="".join(ln.rstrip() + "\n" for ln in no_mask))
            _assert_files(got, exp, name + " vs the reference")
            print("golden case %s: every line taken or faulted for its phase mask, equal to the reference's files" % name)
        elif goldenlib.is_special(name):
            # the rows of the subjects taken, against the reference's rows of the same subjects
            sids = {x[0] for x in _split(taken)}
            for k in ("umug", "umug_pops", "pmug", "pmug_pops"):
                want = "".join(r for r in exp[k].splitlines(True) if r.split(",")[0] in sids)
                assert got[k] == want, (name, k)
            print("golden case %s: the rows of the %d subjects taken equal the reference's" % (name, len(sids)))
    finally:
        g.close()


# --------------------------------------------------------------------------- ambiguity at every scale
def test_c4_messy_and_heavy_subjects():
    conf = _readme_conf()
    g, imp = _graph(conf)
    try:
        tab = synth.Table(open(conf["freq_file"]).read())
        lines = synth.messy_subjects(tab, 3000, 31, max_amb=6, races=["CAU,CAU"])
        _got, res, taken = _compare(imp, lines, "C4 messy")
        assert len(taken) == len(lines) and (_np(res.status) == 0).any()
        assert res.capacity_reruns == 0, "the first result arrays of an ambiguous batch were too small"
        heavy = synth.heavy_subjects(tab, 208, 44, races=["CAU,CAU"])
        longest = max(len(side.split("/")) for ln in heavy for loc in ln.split(",")[1].split("^") for side in loc.split("+"))
        assert longest >= 40
        _got, _res, taken = _compare(imp, heavy, "C4 heavy")
        assert len(taken) == len(heavy)
    finally:
        g.close()


def test_wide_subjects_with_and_without_the_cooperative_slot_pass(monkeypatch):
    conf = _readme_conf()
    tab = synth.Table(open(conf["freq_file"]).read())
    lines = synth.wide_subjects(tab, 16, 45, races=["CAU,CAU"])
    for group in ("4096", "0"):
        monkeypatch.setenv("GRIMB_GROUP_SUBJECTS", group)      # read when an engine is created
        g, imp = _graph(conf)
        try:
            _compare(imp, lines, "wide subjects (slot pass %s)" % ("on" if group != "0" else "off"))
        finally:
            g.close()


def _pop21_conf(tmpdir_name):
    cau = open(os.path.join(goldenlib.GOLD, "data", "cau_hpf.csv")).read()
    pops = ["P%02d" % i for i in range(21)]
    hpf, ctext = synth.multipop_hpf(cau, pops, 121)
    paths = [os.path.join(tmpdir_name, n) for n in ("hpf.csv", "cnt.txt")]
    open(paths[0], "w").write(hpf)
    open(paths[1], "w").write(ctext)
    conf = _readme_conf()
    conf.update({"populations": pops, "UNK_priors": "MR", "number_of_pop_results": 100, "freq_file": paths[0],
                 "pops_count_file": paths[1], "use_pops_count_file": True})
    return conf, synth.Table(hpf, "P00"), synth.race_fields(pops)


@pytest.mark.parametrize("kw", [1, 2], ids=["keys64", "keys128"])
def test_twenty_one_populations_ambiguous(kw, monkeypatch, tmp_path):
    conf, tab, races = _pop21_conf(str(tmp_path))
    g, imp = _graph(conf, monkeypatch, kw)
    try:
        assert g.kw == kw
        lines = synth.messy_subjects(tab, 300, 6, max_amb=4, races=races) + synth.typed_subjects(tab, 200, 3, races)
        _got, res, _taken = _compare(imp, lines, "P = 21 (%d-bit keys)" % (64 * kw))
        assert len(_np(res.umug_pops)) > 0
    finally:
        g.close()


def test_nine_loci_wide_keys(monkeypatch):
    _t, conf, lines, _e = goldenlib.load_case("g6_nine_loci")
    g, imp = _graph(conf, monkeypatch, 2)
    try:
        assert imp.L == 9 and g.kw == 2
        tab = synth.Table(open(conf["freq_file"]).read(), loci=imp.loci)
        lines = lines + synth.messy_subjects(tab, 120, 9, max_amb=4) + synth.typed_subjects(tab, 60, 9)
        _compare(imp, lines, "nine loci, 128-bit keys")
    finally:
        g.close()


def test_plan_a_matrix():
    """planb off: the list route equals the text route, and a typed-locus pattern that is no matrix row comes back
    SKIPPED with the problem flag; planb on: the NotImplementedError of both routes."""
    _t, conf, _lines, _exp = goldenlib.load_case("g8_plan_a_blocks")
    conf["planb"] = False
    g, imp = _graph(conf)
    try:
        tab = synth.Table(open(conf["freq_file"]).read())
        _compare(imp, synth.messy_subjects(tab, 300, 8, max_amb=4, p_missing=0.3), "Plan_A_Matrix, planb off")
        # typed-locus patterns applied on the device (the host tokeniser sends non-matrix lines to the text path)
        full = synth.messy_subjects(tab, 60, 18, max_amb=3, p_missing=0.0, p_unknown=0.0)
        lists = _lists(*_encode_lines(imp, full)[:2])
        subs = [[0, 1, 2, 3, 4], [0, 1], [2, 3, 4], [0, 2], [1, 3], [0, 1, 2]]
        masks = []
        for s in range(len(full)):
            sub = subs[s % len(subs)]
            lists[s] = [sides if l in sub else [[], []] for l, sides in enumerate(lists[s])]
            masks.append(sum(1 << l for l in sub))
        res = imp.impute_genotype_lists(*_flatten(lists, imp.L))
        st, fl = _np(res.status), _np(res.flags)
        for s, m in enumerate(masks):
            assert (st[s] == ST_SKIPPED) == (not imp.type_allowed[m]), (s, m)
            assert bool(fl[s] & 4) == (st[s] == ST_SKIPPED)
            if st[s] == ST_SKIPPED:
                _no_rows(res, s)
        assert (st == ST_SKIPPED).any() and (st != ST_SKIPPED).any()
        imp.cfg.planb = 1
        imp.config["planb"] = True
        lines = synth.messy_subjects(tab, 200, 8, max_amb=2, p_missing=0.0, p_random=0.5)
        with pytest.raises(NotImplementedError, match="Plan_A_Matrix"):
            _lists_run(imp, lines)
    finally:
        g.close()


# --------------------------------------------------------------------------- the encoder's contract
def _encode_lines(imp, lines):
    counts, alleles, unknown, tp = imp.encode_genotype_lists([ln.rstrip().split(",")[1] for ln in lines])
    assert not tp
    return counts, alleles, unknown


def _lists(counts, alleles):
    """counts, alleles -> per subject, per locus, per side: the id lists."""
    out, k = [], 0
    for s in range(counts.shape[0]):
        subj = []
        for l in range(counts.shape[1]):
            sides = []
            for x in range(2):
                n = int(counts[s, l, x])
                sides.append([int(v) for v in alleles[k:k + n]])
                k += n
            subj.append(sides)
        out.append(subj)
    return out


def _flatten(lists, L):
    counts = np.zeros((len(lists), L, 2), np.uint16)
    flat = []
    for s, subj in enumerate(lists):
        for l, sides in enumerate(subj):
            for x, ids in enumerate(sides):
                counts[s, l, x] = len(ids)
                flat.extend(ids)
    return counts, np.array(flat, np.uint16)


def test_duplicate_ids_and_long_lists():
    """Repeated ids inside a side's list (long lists among them: 40+ ids on one side) give the rows of the
    de-duplicated input, and the rows of the text route on GL strings that repeat the same names."""
    conf = _readme_conf()
    g, imp = _graph(conf)
    try:
        tab = synth.Table(open(conf["freq_file"]).read())
        lines = synth.messy_subjects(tab, 150, 12, max_amb=4, p_unknown=0.0) + synth.heavy_subjects(tab, 40, 45)
        lines = [ln for ln in lines if "/" in ln]
        counts, alleles, unknown = _encode_lines(imp, lines)
        clean = _lists(counts, alleles)
        rng = np.random.RandomState(5)
        dup, dup_lines = [], []
        for s, ln in enumerate(lines):
            subj = []
            sid, gl = ln.rstrip().split(",")[:2]
            locs = gl.split("^")
            for l, sides in enumerate(clean[s]):
                new = []
                for x, ids in enumerate(sides):
                    ids = list(ids)
                    if ids and rng.rand() < 0.5:
                        for _ in range(rng.randint(1, 4)):
                            j = rng.randint(len(ids))       # a repeat after the id's first occurrence
                            ids.insert(rng.randint(j + 1, len(ids) + 1), ids[j])
                    new.append(ids)
                subj.append(new)
            dup.append(subj)
            # the same repeats by name
            names = []
            for loc in locs:
                l = imp.locus_index[loc.split("*")[0]]
                halves = []
                for x, side in enumerate(loc.split("+")):
                    by_id = {i: n for i, n in zip(clean[s][l][x], side.split("/"))}
                    halves.append("/".join(by_id[i] for i in dup[s][l][x]))
                names.append("+".join(halves))
            dup_lines.append(sid + "," + "^".join(names) + "\n")
        assert max(len(ids) for subj in dup for sides in subj for ids in sides) >= 40
        dcounts, dalleles = _flatten(dup, imp.L)
        assert len(dalleles) > len(alleles)
        base = imp.impute_genotype_lists(counts, alleles)
        _same(base, imp.impute_genotype_lists(dcounts, dalleles))
        got = render_lists(imp.impute_genotype_lists(dcounts, dalleles), imp, [ln.split(",")[0] for ln in lines],
                           dup_lines, unknown)
        _assert_files(got, _text(imp, dup_lines), "repeated ids")
    finally:
        g.close()


def test_skip_conditions():
    conf = _readme_conf()
    g, imp = _graph(conf)
    try:
        tab = synth.Table(open(conf["freq_file"]).read())
        lines = synth.messy_subjects(tab, 12, 13, max_amb=3, p_missing=0.0, p_unknown=0.0)
        counts, alleles, _u = _encode_lines(imp, lines)
        lists = _lists(counts, alleles)
        lists[1][2][1] = []                                  # exactly one side of a locus lists nothing
        lists[3][0][0][-1] = 0                               # an id 0 inside a list
        lists[5][1][1][0] = 1 << g.key_bits[1]               # an id wider than its locus's key field
        lists[7] = [[[], []] for _ in range(imp.L)]          # no typed locus
        res = imp.impute_genotype_lists(*_flatten(lists, imp.L))
        st, fl = _np(res.status), _np(res.flags)
        for s in range(12):
            if s in (1, 3, 5, 7):
                assert st[s] == ST_SKIPPED and fl[s] & 4, s
                _no_rows(res, s)
            else:
                assert st[s] == 0, s
    finally:
        g.close()


def test_count_sum_mismatch_is_refused_before_alleles_are_read():
    import torch
    from grim.imputation import _lib
    conf = _readme_conf()
    g, imp = _graph(conf)
    try:
        tab = synth.Table(open(conf["freq_file"]).read())
        counts, alleles, _u = _encode_lines(imp, synth.messy_subjects(tab, 20, 14, max_amb=3))
        for bad in (alleles[:-1], np.concatenate([alleles, alleles[:3]])):
            with pytest.raises(RuntimeError, match="n_alleles"):
                imp.impute_genotype_lists(counts, bad)
        # directly: the counts list more ids than the 4-element array holds -- refused after the count pass and
        # its scan (two launches), before any kernel reads `alleles`
        dev = torch.device("cuda", g.device)
        eng = g.engine(imp.workspaces[0])
        d_counts = torch.from_numpy(counts.view(np.int16)).to(dev)
        d_alleles = torch.from_numpy(alleles[:4].view(np.int16)).to(dev)
        priors = torch.ones((1, 1, 1), dtype=torch.float64, device=dev)
        b = _lib.Batch()
        n0 = g.lib.grimb_engine_launches(eng)
        rc = g.lib.grimb_batch_from_genotype_lists(eng, d_counts.data_ptr(), d_alleles.data_ptr(), 4, counts.shape[0], None,
                                                   priors.data_ptr(), 1, None, None, C.byref(b), None)
        assert rc == E_ARG
        assert g.lib.grimb_engine_launches(eng) - n0 == 2
    finally:
        g.close()


def test_sizes_inputs_capacity_growth_and_workspace_reissue():
    import torch
    conf = _readme_conf()
    g, imp = _graph(conf)
    try:
        tab = synth.Table(open(conf["freq_file"]).read())
        lines = synth.messy_subjects(tab, 301, 21, max_amb=5, p_missing=0.3, p_random=0.3)
        counts, alleles, _u = _encode_lines(imp, lines)
        base = imp.impute_genotype_lists(counts, alleles)
        assert base.workspace_retries == 0 and base.pmug_pairs is None
        dev = torch.device("cuda", g.device)
        on_dev = imp.impute_genotype_lists(torch.from_numpy(counts).to(dev), torch.from_numpy(alleles).to(dev))
        assert on_dev.status.is_cuda and on_dev.umug.is_cuda and on_dev.umug.dtype == torch.uint16
        _same(base, on_dev)
        imp._row_caps = (1, 1, 1, 1)                       # GRIMB_E_CAPACITY, then growth
        _same(base, imp.impute_genotype_lists(counts, alleles))
        del imp._row_caps
        imp.workspaces = [1 << 16] + imp.workspaces         # a first tier too small for some subjects
        tiny = imp.impute_genotype_lists(counts, alleles)
        assert tiny.workspace_retries > 0
        _same(base, tiny, pair_evals=False)                # the overflowed first attempts add evaluations
        imp.workspaces = imp.workspaces[1:]
        empty = imp.impute_genotype_lists(counts[:0], alleles[:0])
        assert len(empty) == 0 and len(empty.umug_off) == 1 and len(empty.umug) == 0
        untyped = imp.impute_genotype_lists(np.zeros((4, imp.L, 2), np.uint16), alleles[:0])
        assert (untyped.status == ST_SKIPPED).all() and len(untyped.pmug) == 0
        n_in = counts.astype(np.int64).sum((1, 2))
        for n in (1, 2, 3, 5, 7, 33):
            part = imp.impute_genotype_lists(counts[:n], alleles[:int(n_in[:n].sum())])
            assert np.array_equal(part.status, base.status[:n])
            for k in KINDS:
                o = getattr(base, k + "_off")
                assert np.array_equal(getattr(part, k), getattr(base, k)[:o[n]]), (n, k)
                assert getattr(part, k + "_prob").tobytes() == getattr(base, k + "_prob")[:o[n]].tobytes(), (n, k)
    finally:
        g.close()


# --------------------------------------------------------------------------- typed subjects are unchanged
def _p1_conf(tmp_path):
    names, fa, f = synth.zipf_arrays(3000, [60, 90, 50, 30, 60], 5, synth.LOCI5)
    hpf = os.path.join(str(tmp_path), "p1_hpf.csv")
    with open(hpf, "w") as fh:
        fh.write("hap,pop,freq\n")
        for i in range(len(fa)):
            fh.write("%s,CAU,%r\n" % ("~".join(names[l][fa[i, l] - 1] for l in range(5)), float(f[i])))
    conf = _readme_conf()
    conf.update({"freq_file": hpf, "freq_trim_threshold": 1e-30})
    return conf, names, fa, f


@pytest.mark.parametrize("table", ["readme", "p1"])
def test_typed_subjects_equal_the_dense_route(table, tmp_path):
    """Every count 1: the same per-subject arrays and rows, bit for bit, as impute_genotypes; on the P = 1 table
    the general form of k_fast_probe serves them (kernel_ms 6 == 0)."""
    if table == "readme":
        conf = _readme_conf()
        tab = synth.Table(open(conf["freq_file"]).read())
        lines = synth.typed_subjects(tab, 2000, 3)
    else:
        conf, names, fa, f = _p1_conf(tmp_path)
        lines = synth.array_subject_lines(names, fa, f, 4001, 7)
    g, imp = _graph(conf)
    try:
        gls = [ln.rstrip().split(",")[1] for ln in lines]
        ids, _u, tp = imp.encode_genotypes(gls)
        counts, alleles, _u2, tp2 = imp.encode_genotype_lists(gls)
        assert not tp and not tp2 and (counts == 1).all()
        dense = imp.impute_genotypes(ids)
        lists = imp.impute_genotype_lists(counts, alleles)
        _same(dense, lists, pair_evals=False)
        if table == "p1":
            assert g.lib.grimb_engine_kernel_ms(g.engine(imp.workspaces[0]), 6) == 0
    finally:
        g.close()


def test_mixed_batch_rows_of_simple_and_typed_records(tmp_path):
    """80 % typed, 20 % ambiguous in one lists batch (non-NULL counts): k_rows_fill reads the SIMPLE records of the
    typed subjects from the general form, and the rows equal the text route."""
    conf, names, fa, f = _p1_conf(tmp_path)
    g, imp = _graph(conf)
    try:
        tab = synth.Table(open(conf["freq_file"]).read())
        typed = synth.array_subject_lines(names, fa, f, 1600, 8, variants=False)
        messy = synth.messy_subjects(tab, 400, 9, max_amb=4)
        lines = [ln for pair in zip(typed[0::4], typed[1::4], typed[2::4], typed[3::4], messy) for ln in pair]
        got, res, taken = _lists_run(imp, lines)
        assert g.lib.grimb_engine_kernel_ms(g.engine(imp.workspaces[0]), 6) == 0
        assert len(taken) == len(lines)
        _assert_files(got, _text(imp, taken), "mixed batch")
    finally:
        g.close()


# --------------------------------------------------------------------------- phase masks
def test_random_phase_masks(tmp_path):
    _t, conf, _lines, _exp = goldenlib.load_case("g7_phase_masks")
    conf.pop("_hap_pop_pair")
    tab = synth.Table(open(conf["freq_file"]).read(), "AAA")
    L = len(conf["loci_map"])
    lines = synth.messy_subjects(tab, 400, 17, max_amb=4, races=synth.race_fields(["AAA", "BBB", "CCC"]))
    rng = np.random.RandomState(17)
    masks = {}
    for s, ln in enumerate(lines):
        sid = ln.split(",")[0]
        kind = s % 5
        if kind == 0:
            bits = [0] * L
        elif kind == 1:
            bits = [1] * 16                               # 0xFFFF
        elif kind == 2:
            bits = [0] * L
            bits[rng.randint(len(bits))] = 1              # a single bit
        elif kind == 3:
            bits = [int(x) for x in rng.randint(0, 2, L)]
        else:
            continue                                       # no entry: the text path faults the line
        masks[sid] = bits
    path = os.path.join(str(tmp_path), "masks.json")
    with open(path, "w") as f:
        json.dump(masks, f)
    conf["bin_imputation_in_file"] = path
    g, imp = _graph(conf)
    try:
        sids = [ln.split(",")[0] for ln in lines]
        pm, missing = imp.phase_masks_for(sids)
        assert missing == [s for s in range(len(lines)) if s % 5 == 4]
        assert pm[0] == 0 and pm[1] == 0xFFFF and bin(int(pm[2])).count("1") == 1
        _got, _res, taken = _compare(imp, lines, "random phase masks")
        assert len(taken) == len(lines) - len(missing)
        with pytest.raises(ValueError, match="phase_masks_for"):
            imp.impute_genotype_lists(np.zeros((1, imp.L, 2), np.uint16), np.zeros(0, np.uint16))
    finally:
        g.close()


# --------------------------------------------------------------------------- hap_pop_pair and em
def test_hap_pop_pair_twenty_one_populations(tmp_path):
    conf, tab, races = _pop21_conf(str(tmp_path))
    g, imp = _graph(conf)
    try:
        lines = synth.messy_subjects(tab, 300, 23, max_amb=4, races=races) + synth.typed_subjects(tab, 100, 24, races)
        got, res, taken = _lists_run(imp, lines, em_mr=True)
        assert imp.cfg.hap_pop_pair == 0                   # the mode applied to that call only
        assert res.pmug_pairs is not None and tuple(res.pmug_pairs.shape) == (res.pmug.shape[0], 2)
        assert len(set(_np(res.pmug_pairs).reshape(-1).tolist())) > 2
        _assert_files(got, _text(imp, taken, em_mr=True), "hap_pop_pair, P = 21")
        # workspace re-issue under em_mr: the re-issued subjects' pmug_pairs are spliced back in input order
        counts, alleles, _u = _encode_lines(imp, taken)
        pri = [imp.prior_index(*x[2:]) for x in _split(taken)]
        base = imp.impute_genotype_lists(counts, alleles, pri, em_mr=True)
        imp.workspaces = [1 << 16] + imp.workspaces
        tiny = imp.impute_genotype_lists(counts, alleles, pri, em_mr=True)
        imp.workspaces = imp.workspaces[1:]
        assert tiny.workspace_retries > 0
        _same(base, tiny, pair_evals=False)
    finally:
        g.close()


def test_rows_refuse_hap_pop_pair_without_pmug_pairs():
    from grim.imputation import _lib
    g, imp = _graph(_readme_conf())
    try:
        cfg = _lib.Config()
        C.pointer(cfg)[0] = imp.cfg
        cfg.hap_pop_pair = 1
        tot = np.zeros(4, np.int64)
        rows = _lib.Rows()
        rows.totals = tot.ctypes.data
        rc = g.lib.grimb_results_rows(g.engine(imp.workspaces[0]), C.byref(cfg), C.byref(_lib.Batch()),
                                      C.byref(_lib.Results()), C.byref(rows), None)
        assert rc == E_ARG
    finally:
        g.close()


def test_em_mode():
    """em = no Plan C for the haplotype output: equal to impute_lines(em=True) on subjects that reach Plan C, and
    different from em=False on at least one of them."""
    conf = _readme_conf()
    g, imp = _graph(conf)
    try:
        tab = synth.Table(open(conf["freq_file"]).read())
        lines = synth.messy_subjects(tab, 400, 11, max_amb=3, p_missing=0.3, p_random=0.3)
        got, res, _taken = _compare(imp, lines, "em", em=True)
        plain, _res, _t = _lists_run(imp, lines)
        assert 3 in set(_np(res.plan_umug).tolist())
        assert any(got[k] != plain[k] for k in goldenlib.KEYS), "em changed no output"
    finally:
        g.close()
