"""GPU: the device-resident genotype interface (Imputation.encode_genotypes / impute_genotypes: genotype tensor ->
grimb_batch_from_genotypes -> the imputation kernels -> grimb_results_rows -> ragged row tensors).  A test-only
renderer turns the rows into the six output texts (str(float), sorted .umug.pops names, all_pops, the Plan C `0`
population row), and every case compares them byte for byte with impute_text on the same lines -- and, where
every line of a golden case is an unambiguous genotype, with the reference's own output files.  The cases cover
the packed batch form (k_fast_probe2), the general form (missing loci, Plan B / C, GENERAL records), TYPED records
with pair codes, four and nine loci, 128-bit keys, a Plan_A_Matrix, invalid rows, row-capacity growth, workspace
re-issue, batch sizes, numpy against CUDA input, the unsupported modes, and the benchmark's own batch."""
import json
import os

import numpy as np
import pytest

import goldenlib
import synth

pytestmark = pytest.mark.gpu

ST_SKIPPED = 4


def _graph(conf, monkeypatch=None, kw=None):
    from grim.imputation.impute import Imputation
    from grim.imputation.networkx_graph import Graph
    from grim.run_impute_def import load_config
    if kw is not None:
        monkeypatch.setenv("GRIMB_KEY_WORDS", str(kw))
    cfg = load_config(conf)
    g = Graph(cfg).build_graph()
    return g, Imputation(g, cfg)


def _split(lines):
    """-> (sid, gl, race1, race2) per line, as the line parser of impute.py reads it; None for lines it rejects."""
    out = []
    for raw in lines:
        raw = raw.rstrip()
        f = raw.split(",") if "," in raw else raw.split("%")
        if len(f) < 2 or len(f) == 3:
            out.append(None)
            continue
        out.append((f[0], f[1], f[2] if len(f) > 2 else None, f[3] if len(f) > 2 else None))
    return out


def _to_np(x):
    """numpy view of a result array (CUDA tensors of unsigned types go through their signed twins)."""
    if not hasattr(x, "cpu"):
        return x
    import torch
    signed = {torch.uint16: (torch.int16, np.uint16), torch.uint32: (torch.int32, np.uint32)}
    if x.dtype in signed:
        return x.view(signed[x.dtype][0]).cpu().numpy().view(signed[x.dtype][1])
    return x.cpu().numpy()


def render(res, imp, sids, raws, unknown):
    """The six output texts of impute_text, from the rows of impute_genotypes (test-only renderer)."""
    conf = imp.config
    L = imp.L
    g = {k: _to_np(getattr(res, k)) for k in ("status", "flags", "plan_umug", "tot_umug")}
    rows = {}
    for k in ("umug", "pmug", "umug_pops", "pmug_pops"):
        rows[k] = (_to_np(getattr(res, k)).astype(np.int64), _to_np(getattr(res, k + "_prob")), _to_np(getattr(res, k + "_off")))
    files = {k: [] for k in goldenlib.KEYS}

    def name(s, l, i):
        al = res.alleles[l]
        return al[i - 1] if 1 <= i <= len(al) else unknown[s][(l, i)]

    def pop(p):
        return "all_pops" if p == 0xFFFF else res.populations[p]

    for s, sid in enumerate(sids):
        fl = int(g["flags"][s])
        if fl & 4:
            files["problem"].append("%d,%s\n" % (s, sid) if g["status"][s] == ST_SKIPPED else raws[s].rstrip() + "\n")
            continue
        if fl & 2:
            files["miss"].append("%d,%s\n" % (s, sid))
        if conf["output_haplotypes"]:
            r, p, o = rows["pmug"]
            for k, q in enumerate(range(o[s], o[s + 1])):
                h = ["~".join(name(s, l, int(r[q, x, l])) for l in range(L) if r[q, x, l]) for x in (0, 1)]
                files["pmug"].append("%s,%s+%s,%r,%d\n" % (sid, h[0], h[1], float(p[q]), k))
            r, p, o = rows["pmug_pops"]
            for k, q in enumerate(range(o[s], o[s + 1])):
                files["pmug_pops"].append("%s,%s,%s,%r,%d\n" % (sid, pop(r[q, 0]), pop(r[q, 1]), float(p[q]), k))
        if conf["output_MUUG"]:
            r, p, o = rows["umug"]
            for k, q in enumerate(range(o[s], o[s + 1])):
                geno = "^".join("+".join(sorted([name(s, l, int(r[q, l, 0])), name(s, l, int(r[q, l, 1]))]))
                                for l in range(L) if r[q, l, 0])
                files["umug"].append("%s,%s,%r,%d\n" % (sid, geno, float(p[q]), k))
            r, p, o = rows["umug_pops"]
            planc_empty = g["plan_umug"][s] == 3 and g["tot_umug"][s] == 0
            for k, q in enumerate(range(o[s], o[s + 1])):
                a, b = sorted([pop(r[q, 0]), pop(r[q, 1])])
                files["umug_pops"].append("%s,%s,%s,%s,%d\n" % (sid, a, b, "0" if planc_empty else repr(float(p[q])), k))
    return {k: "".join(v) for k, v in files.items()}


def _genotype_run(imp, lines, cuda=True):
    """Lines -> (the genotype route's six texts, results, the lines it took).  Lines the encoder sends to the
    text path (ambiguity, problem, fault) and lines the line parser rejects are left out."""
    import torch
    parsed = _split(lines)
    keep = [i for i, x in enumerate(parsed) if x is not None]
    ids, unknown, text_path = imp.encode_genotypes([parsed[i][1] for i in keep])
    ok = [j for j in range(len(keep)) if j not in set(text_path)]
    taken = [lines[keep[j]] for j in ok]
    ids, unknown = ids[ok], [unknown[j] for j in ok]
    pri = [imp.prior_index(parsed[keep[j]][2], parsed[keep[j]][3]) for j in ok]
    x = torch.from_numpy(ids).cuda(imp.netGraph.device) if cuda else ids
    res = imp.impute_genotypes(x, pri)
    sids = [parsed[keep[j]][0] for j in ok]
    return render(res, imp, sids, taken, unknown), res, taken


def _text(imp, lines):
    out = imp.impute_text("".join(lines).encode("utf8"))
    return {k: v.decode("utf8") for k, v in out.items()}


def _assert_files(got, want, what):
    for k in goldenlib.KEYS:
        if got[k] != want[k]:
            a, b = got[k].splitlines(), want[k].splitlines()
            i = next((j for j in range(min(len(a), len(b))) if a[j] != b[j]), min(len(a), len(b)))
            raise AssertionError("%s: %s differs at row %d: %r vs %r (%d / %d rows)" % (
                what, k, i, a[i] if i < len(a) else None, b[i] if i < len(b) else None, len(a), len(b)))


def _compare(imp, lines, what, cuda=True):
    got, res, taken = _genotype_run(imp, lines, cuda)
    _assert_files(got, _text(imp, taken), what)
    return got, res, taken


# --------------------------------------------------------------------------- golden cases (every configuration)
@pytest.mark.parametrize("name", goldenlib.text_case_names())
def test_golden_case_through_the_genotype_route(name, monkeypatch):
    _t, conf, lines, exp = goldenlib.load_case(name)
    if conf.get("Plan_A_Matrix"):
        conf["planb"] = False    # under a matrix the reference's Plan B is not defined (DESIGN 7)
    g, imp = _graph(conf)
    try:
        got, res, taken = _compare(imp, lines, name)
        eng = g.engine(imp.workspaces[0])
        if taken:
            assert g.lib.grimb_engine_kernel_ms(eng, 7) >= 0 and g.lib.grimb_engine_kernel_ms(eng, 8) >= 0
        if len(taken) == len(lines) and not conf.get("Plan_A_Matrix"):
            _assert_files(got, exp, name + " vs the reference")
    finally:
        g.close()


def test_plan_a_matrix_with_planb_raises():
    """Under a Plan_A_Matrix with planb on, a subject that leaves Plan A without a result raises on both routes."""
    _t, conf, _lines, _exp = goldenlib.load_case("g8_plan_a_blocks")
    conf["planb"] = True
    g, imp = _graph(conf)
    try:
        tab = synth.Table(open(conf["freq_file"]).read())
        lines = synth.messy_subjects(tab, 200, 8, max_amb=1, p_missing=0.0, p_random=0.5)
        with pytest.raises(NotImplementedError):
            _text(imp, lines)
        with pytest.raises(NotImplementedError, match="Plan_A_Matrix"):
            _genotype_run(imp, lines)
    finally:
        g.close()


def test_plan_a_matrix_rejects_non_matrix_patterns():
    """The encoder applies type_allowed on the device: a typed-locus pattern that is no matrix row comes back
    SKIPPED with the problem flag (the text path writes "i,id" to .problem for it)."""
    _t, conf, _lines, _exp = goldenlib.load_case("g8_plan_a_blocks")
    conf["planb"] = False
    g, imp = _graph(conf)
    try:
        assert imp.loci == synth.LOCI5
        tab = synth.Table(open(conf["freq_file"]).read())
        subs = [[0, 1, 2, 3, 4], [0, 1], [2, 3, 4], [0, 2], [1, 3], [0, 1, 2]]
        full = synth.typed_subjects(tab, 60, 3)
        ids, unknown, tp = imp.encode_genotypes([ln.rstrip().split(",")[1] for ln in full])
        assert not tp
        lines, sids, masks = [], [], []
        for s, ln in enumerate(full):
            sid, gl = ln.rstrip().split(",")[:2]
            sub = subs[s % len(subs)]
            for l in range(imp.L):
                if l not in sub:
                    ids[s, l] = 0
            lines.append(sid + "," + "^".join(gl.split("^")[l] for l in sub) + "\n")
            sids.append(sid)
            masks.append(sum(1 << l for l in sub))
        res = imp.impute_genotypes(ids)
        _assert_files(render(res, imp, sids, lines, unknown), _text(imp, lines), "Plan_A_Matrix patterns")
        st, fl = res.status, res.flags
        for s, m in enumerate(masks):
            assert (st[s] == ST_SKIPPED) == (not imp.type_allowed[m]), (s, m)
            assert bool(fl[s] & 4) == (st[s] == ST_SKIPPED)
        assert (st == ST_SKIPPED).any() and (st != ST_SKIPPED).any()
    finally:
        g.close()


# --------------------------------------------------------------------------- synthetic tables
def _readme_conf():
    _t, conf, _l, _e = goldenlib.load_case("g1_readme_donor")
    return conf


def test_packed_form_single_population(monkeypatch):
    """Fully typed P = 1 batch: the packed form and k_fast_probe2, with homozygous, unknown-allele and
    recombinant subjects (hand-over to the general kernel) and a batch size that is no multiple of 4."""
    names, fa, f = synth.zipf_arrays(3000, [60, 90, 50, 30, 60], 5, synth.LOCI5)
    d = os.environ.get("TMPDIR", "/tmp")
    hpf = os.path.join(d, "geno_api_%d_hpf.csv" % os.getpid())
    with open(hpf, "w") as fh:
        fh.write("hap,pop,freq\n")
        for i in range(len(fa)):
            fh.write("%s,CAU,%r\n" % ("~".join(names[l][fa[i, l] - 1] for l in range(5)), float(f[i])))
    conf = _readme_conf()
    conf.update({"freq_file": hpf, "freq_trim_threshold": 1e-30})
    g, imp = _graph(conf)
    try:
        lines = synth.array_subject_lines(names, fa, f, 4001, 7)
        _got, res, taken = _compare(imp, lines, "packed P = 1")
        eng = g.engine(imp.workspaces[0])
        assert g.lib.grimb_engine_kernel_ms(eng, 6) == 2, "the packed batch did not run k_fast_probe2"
        assert len(taken) == len(lines)
    finally:
        g.close()
        os.unlink(hpf)


def test_general_form_missing_loci_plan_b_and_c():
    conf = _readme_conf()
    g, imp = _graph(conf)
    try:
        tab = synth.Table(open(conf["freq_file"]).read())
        lines = synth.messy_subjects(tab, 400, 11, max_amb=1, p_missing=0.3, p_random=0.3)
        lines.append("D1,A*01:01+A*02:01^B*08:01+B*44:02\n")       # the README donor: typed at A and B
        _got, res, taken = _compare(imp, lines, "general form")
        eng = g.engine(imp.workspaces[0])
        assert g.lib.grimb_engine_kernel_ms(eng, 6) != 2
        plans = set(_to_np(res.plan_umug).tolist())
        assert {2, 3} <= plans, "Plan B and Plan C subjects expected, got plans %r" % plans
        assert len(taken) == len(lines)
    finally:
        g.close()


@pytest.mark.parametrize("kw", [1, 2], ids=["keys64", "keys128"])
def test_twenty_one_populations_typed_records(kw, monkeypatch):
    cau = open(os.path.join(goldenlib.GOLD, "data", "cau_hpf.csv")).read()
    pops = ["P%02d" % i for i in range(21)]
    hpf, ctext = synth.multipop_hpf(cau, pops, 121)
    d = os.environ.get("TMPDIR", "/tmp")
    paths = [os.path.join(d, "geno_api_%d_%s" % (os.getpid(), n)) for n in ("hpf.csv", "cnt.txt")]
    open(paths[0], "w").write(hpf)
    open(paths[1], "w").write(ctext)
    conf = _readme_conf()
    conf.update({"populations": pops, "UNK_priors": "MR", "number_of_pop_results": 100, "freq_file": paths[0],
                 "pops_count_file": paths[1], "use_pops_count_file": True})
    g, imp = _graph(conf, monkeypatch, kw)
    try:
        assert g.kw == kw
        tab = synth.Table(hpf, "P00")
        races = synth.race_fields(pops)
        lines = synth.typed_subjects(tab, 500, 3, races)
        lines += synth.messy_subjects(tab, 100, 6, max_amb=1, races=races)
        _got, res, _taken = _compare(imp, lines, "P = 21 (%d-bit keys)" % (64 * kw))
        assert len(_to_np(res.umug_pops)) > 0
    finally:
        g.close()
        for p in paths:
            os.unlink(p)


def test_four_loci(tmp_path):
    loci = ["A", "B", "C", "DRB1"]
    hpf = synth.zipf_table(300, [5, 6, 4, 5], 26, loci=loci)
    open(os.path.join(str(tmp_path), "hpf.csv"), "w").write(hpf)
    conf = _readme_conf()
    conf.update({"freq_file": os.path.join(str(tmp_path), "hpf.csv"), "freq_trim_threshold": 1e-30,
                 "loci_map": {"A": 1, "B": 2, "C": 3, "DRB1": 4},
                 "Plan_B_Matrix": [[[1, 2, 3, 4]], [[1, 2], [3, 4]], [[1], [2], [3], [4]]]})
    g, imp = _graph(conf)
    try:
        assert imp.L == 4
        tab = synth.Table(hpf, loci=loci)
        lines = synth.typed_subjects(tab, 301, 4) + synth.messy_subjects(tab, 100, 4, max_amb=1)
        _compare(imp, lines, "four loci")
    finally:
        g.close()


def test_nine_loci_wide_keys(monkeypatch):
    _t, conf, lines, _e = goldenlib.load_case("g6_nine_loci")
    g, imp = _graph(conf, monkeypatch, 2)
    try:
        assert imp.L == 9 and g.kw == 2
        tab = synth.Table(open(conf["freq_file"]).read(), loci=imp.loci)
        lines = lines + synth.typed_subjects(tab, 200, 9) + synth.messy_subjects(tab, 60, 9, max_amb=1)
        _compare(imp, lines, "nine loci, 128-bit keys")
    finally:
        g.close()


# --------------------------------------------------------------------------- input handling and the call's contract
def test_invalid_rows_come_back_skipped():
    g, imp = _graph(_readme_conf())
    try:
        L = imp.L
        tab = synth.Table(open(imp.config["freq_file"]).read())
        ids, _u, tp = imp.encode_genotypes([ln.split(",")[1] for ln in synth.typed_subjects(tab, 9, 1)])
        assert not tp
        ids[1, 2, 1] = 0                                   # one side of a locus 0
        ids[3, 0, 0] = (1 << g.key_bits[0])                # an id past its locus's key field
        ids[5] = 0                                         # no typed locus
        res = imp.impute_genotypes(ids)
        st, fl = res.status, res.flags
        for s in (1, 3, 5):
            assert st[s] == ST_SKIPPED and fl[s] & 4
            for k in ("umug", "pmug", "umug_pops", "pmug_pops"):
                o = getattr(res, k + "_off")
                assert o[s + 1] == o[s]
        assert all(st[s] == 0 for s in (0, 2, 4, 6, 7, 8))
        assert res.umug.shape[1:] == (L, 2) and res.pmug.shape[1:] == (2, L)
    finally:
        g.close()


def _same(a, b):
    for k in ("status", "flags", "plan_umug", "plan_pmug", "tot_umug", "tot_pmug"):
        assert np.array_equal(_to_np(getattr(a, k)), _to_np(getattr(b, k))), k
    for k in ("umug", "pmug", "umug_pops", "pmug_pops"):
        for suf in ("", "_off"):
            assert np.array_equal(_to_np(getattr(a, k + suf)), _to_np(getattr(b, k + suf))), k + suf
        assert _to_np(getattr(a, k + "_prob")).tobytes() == _to_np(getattr(b, k + "_prob")).tobytes(), k
    assert a.pair_evals == b.pair_evals


def test_capacity_growth_workspace_reissue_sizes_and_inputs():
    import torch
    conf = _readme_conf()
    g, imp = _graph(conf)
    try:
        tab = synth.Table(open(conf["freq_file"]).read())
        lines = synth.messy_subjects(tab, 301, 21, max_amb=1, p_missing=0.3, p_random=0.3)
        ids, _u, tp = imp.encode_genotypes([ln.split(",")[1] for ln in lines])
        base = imp.impute_genotypes(ids)
        assert base.workspace_retries == 0
        on_dev = imp.impute_genotypes(torch.from_numpy(ids).cuda(g.device))
        assert on_dev.status.is_cuda and on_dev.umug.is_cuda and on_dev.umug.dtype == torch.uint16
        _same(base, on_dev)
        imp._row_caps = (1, 1, 1, 1)                       # GRIMB_E_CAPACITY, then growth
        _same(base, imp.impute_genotypes(ids))
        del imp._row_caps
        imp.workspaces = [1 << 16] + imp.workspaces         # a first tier too small for some subjects
        tiny = imp.impute_genotypes(ids)
        assert tiny.workspace_retries > 0
        tiny.pair_evals = base.pair_evals                  # the overflowed first attempts add evaluations
        _same(base, tiny)
        imp.workspaces = imp.workspaces[1:]
        empty = imp.impute_genotypes(ids[:0])
        assert len(empty) == 0 and len(empty.umug_off) == 1 and len(empty.umug) == 0
        for n in (1, 2, 3, 5, 7):
            part = imp.impute_genotypes(ids[:n])
            assert np.array_equal(part.status, base.status[:n])
            o = base.umug_off
            assert np.array_equal(part.umug, base.umug[:o[n]])
    finally:
        g.close()


def test_unsupported_modes_raise():
    g, imp = _graph(_readme_conf())
    try:
        ids = np.zeros((2, imp.L, 2), np.uint16)
        for kw in ({"em_mr": True}, {"em": True}):
            with pytest.raises(NotImplementedError, match="em"):
                imp.impute_genotypes(ids, **kw)
        imp.cfg.encounter_order = 1
        with pytest.raises(NotImplementedError, match="encounter_order"):
            imp.impute_genotypes(ids)
        imp.cfg.encounter_order = 0
        imp.phase_masks = {}
        with pytest.raises(NotImplementedError, match="bin_imputation_in_file"):
            imp.impute_genotypes(ids)
    finally:
        g.close()


# --------------------------------------------------------------------------- the benchmark's batch
def test_benchmark_batch_rows_equal_the_compact_records():
    """bench.py's table and 2^20 subjects: the row tensors equal a host decode (Imputation._subject_rows) of the
    GrimbCompact records grimb_impute_device returned for the same packed batch (all subjects through vectorised
    arrays, a sample through _subject_rows), and a 20,000-subject sample renders to impute_text byte for byte."""
    import ctypes as C
    import torch
    import bench
    from grim.imputation import _lib
    from grim.imputation.impute import Imputation
    from grim.imputation.networkx_graph import Graph
    from grim.run_impute_def import load_config
    names, fa, ff = bench.make_table(1000000)
    conf = load_config(bench.base_conf())
    g = Graph(conf).from_arrays(names, fa, ff)
    try:
        imp = Imputation(g, conf, np.ones(1))
        S = 1 << 20
        _batch, alleles = bench.make_subjects(fa, ff, S, bench.SUBJECT_SEED)
        dev = torch.device("cuda", g.device)
        res = imp.impute_genotypes(torch.from_numpy(alleles).to(dev))
        eng = g.engine(imp.workspaces[0])
        assert g.lib.grimb_engine_kernel_ms(eng, 6) == 2
        # the existing device route on the packed batch of bench.py
        pk, pf = bench.pack_batch(alleles, g.key_bits, [len(a) for a in names])
        d_pk = torch.from_numpy(pk.view(np.int64)).to(dev)
        d_pf = torch.from_numpy(pf.view(np.int16)).to(dev)
        priors = torch.ones((1, 1, 1), dtype=torch.float64, device=dev)
        b = _lib.Batch()
        b.n_subjects, b.packed_keys, b.packed_flags, b.priors, b.n_priors = S, d_pk.data_ptr(), d_pf.data_ptr(), priors.data_ptr(), 1
        caps = (S * 2, S // 8 + 1024, S // 4 + 1024, S // 4 + 1024)
        out = [torch.zeros(c * sz, dtype=torch.uint8, device=dev) for c, sz in zip((S,) + caps, (16, 8, 48, 24, 16))]
        tot = np.zeros(9, np.int64)
        r = _lib.Results()
        r.compact, r.totals = out[0].data_ptr(), tot.ctypes.data
        r.words, r.word_capacity = out[1].data_ptr(), caps[0]
        r.general, r.general_capacity = out[2].data_ptr(), caps[1]
        r.hap_rows, r.hap_capacity = out[3].data_ptr(), caps[2]
        r.pop_rows, r.pop_capacity = out[4].data_ptr(), caps[3]
        stream = torch.cuda.current_stream(dev)
        _lib.check(g.lib.grimb_impute_device(eng, C.byref(imp.cfg), C.byref(b), C.byref(r), C.c_void_p(stream.cuda_stream)),
                   "grimb_impute_device", g.lib)
        ra = _lib.ResultArrays(S, 1, words=max(16, int(tot[0])), general=max(16, int(tot[1])), hap=max(16, int(tot[2])),
                               pop=max(16, int(tot[3])))
        ra.compact[:] = out[0].cpu().numpy().view(_lib.COMPACT_DTYPE)
        ra.words[:int(tot[0])] = out[1][:int(tot[0]) * 8].cpu().numpy().view(np.uint64)
        ra.general[:int(tot[1])] = out[2][:int(tot[1]) * 48].cpu().numpy().view(_lib.SUBJECT_DTYPE)
        ra.hap_rows[:int(tot[2])] = out[3][:int(tot[2]) * 24].cpu().numpy().view(_lib.hap_row_dtype(1))
        ra.pop_rows[:int(tot[3])] = out[4][:int(tot[3]) * 16].cpu().numpy().view(_lib.POP_ROW_DTYPE)
        assert res.pair_evals == int(tot[4])
        # every subject: status, UMUG probability (= the record's total), PMUG row counts and probabilities
        comp = ra.compact
        st = res.status.cpu().numpy()
        assert np.array_equal(st, comp["status"])
        uo, up = res.umug_off.cpu().numpy(), res.umug_prob.cpu().numpy()
        po, pp = res.pmug_off.cpu().numpy(), res.pmug_prob.cpu().numpy()
        simple = (comp["kind_flags"] & 3) == _lib.KIND_SIMPLE
        has = (comp["kind_flags"] & _lib.KIND_HAS_RESULTS) != 0
        assert np.array_equal(np.diff(uo)[simple], (simple & has)[simple].astype(np.int64))
        assert up[uo[:-1][simple & has]].tobytes() == comp["total"][simple & has].tobytes()
        short = simple & ((comp["kind_flags"] >> 4) != 15)
        assert np.array_equal(np.diff(po)[short], (comp["kind_flags"][short] >> 4).astype(np.int64))
        single = short & ((comp["kind_flags"] & _lib.KIND_WORDS) == 0) & has
        assert pp[po[:-1][single]].tobytes() == comp["total"][single].tobytes()
        # a seeded sample through _subject_rows, row by row
        um, pm = res.umug.cpu().numpy(), res.pmug.cpu().numpy()
        name = lambda l, i: names[l][i - 1]
        sample = np.sort(np.random.RandomState(3).choice(S, 3000, replace=False))
        for s in list(sample) + list(np.nonzero(~short)[0][:200]):
            ids = [int(x) for x in alleles[s].reshape(-1)]
            want = imp._subject_rows(ra, s, ids, None)
            got_u = [([(name(l, int(um[q, l, 0])), name(l, int(um[q, l, 1]))) for l in range(5)], float(up[q]))
                     for q in range(uo[s], uo[s + 1])]
            assert [([tuple(sorted(p)) for p in pairs], pr) for pairs, pr in want["umug"]] == \
                [([tuple(sorted(p)) for p in pairs], pr) for pairs, pr in got_u]
            got_p = [([name(l, int(pm[q, 0, l])) for l in range(5)], [name(l, int(pm[q, 1, l])) for l in range(5)], float(pp[q]))
                     for q in range(po[s], po[s + 1])]
            assert want["pmug"] == got_p
        # a 20,000-subject sample renders to impute_text byte for byte
        lines = bench.subject_lines(names, alleles, 0, 20000)
        sub = imp.impute_genotypes(alleles[:20000])
        got = render(sub, imp, ["S%d" % s for s in range(20000)], lines, [None] * 20000)
        _assert_files(got, _text(imp, lines), "bench batch sample")
    finally:
        g.close()
