"""Host side of the B200 imputation path: class Imputation keeps the reference's name and
entry points (grim/imputation/impute.py:121 `Imputation`, :1985 `impute_file`, :1940
`impute_one` in the reference) but only tokenises GL strings, ships batches through the C ABI
(include/grimb200.h) and formats the packed result rows into the six output files.

Everything numeric happens on the GPU; the one exception is the P x P population prior
(impute.py:1844-1924 of the reference), which depends only on the (race1, race2) fields, is
memoised per distinct pair and computed with the same numpy operation order so it is
bit-identical."""
import ctypes as C
import os
import sys
import time

import numpy as np

from . import _lib

H_OK, H_PROBLEM, H_FAULT = 0, 1, 2   # host-side classification of an input line


def clean_up_gl(gl):
    # same observable behaviour as the reference's clean_up_gl (impute.py:105-118)
    gl = gl.replace("g", "").replace("L", "")
    parts = gl.split("^")
    for bad in [p for p in parts if p.strip("U") != p]:
        parts.remove(bad)
    return "^".join(parts)


def make_config(conf, loci, n_pops):
    """run_impute_def-style config dict -> GrimbConfig."""
    L = len(loci)
    c = _lib.Config()
    c.epsilon = float(conf["epsilon"])
    if not c.epsilon > 0:
        raise ValueError("epsilon must be > 0")
    fmd = conf["factor_missing_data"]
    for k in range(L + 1):
        c.factor_missing_pow[k] = float(fmd ** k)
    c.options_threshold = int(conf["number_of_options_threshold"])
    c.max_haps_in_phase = int(conf["max_haplotypes_number_in_phase"])
    c.n_results = int(conf["number_of_results"])
    c.n_pop_results = int(conf["number_of_pop_results"])
    c.planb = 1 if conf["planb"] else 0
    c.output_umug = 1 if conf["output_MUUG"] else 0
    c.output_pmug = 1 if conf["output_haplotypes"] else 0
    c.save_space = 1 if conf["save_mode"] else 0
    # the reference calls Python's sum() on frequency vectors; CPython >= 3.12 compensates it
    c.compensated_sum = 1 if sys.version_info >= (3, 12) else 0
    matrix = conf["matrix_planb"]
    if len(matrix) > _lib.MAX_ROWS:
        raise NotImplementedError("Plan_B_Matrix has more than %d rows" % _lib.MAX_ROWS)
    all_indices = list(set(range(1, L + 1)))  # impute.py:1118 of the reference
    c.n_rows = len(matrix)
    for r, row in enumerate(matrix):
        if len(row) > _lib.MAX_BLOCKS:
            raise NotImplementedError("Plan_B_Matrix row with more than %d blocks" % _lib.MAX_BLOCKS)
        c.row_blocks[r] = len(row)
        for b, blk in enumerate(row):
            if list(blk) != sorted(blk) or any(i < 1 or i > L for i in blk):
                raise NotImplementedError("Plan_B_Matrix blocks must list loci indices in ascending order")
            m = 0
            for i in blk:
                m |= 1 << (i - 1)
            c.block_mask[r][b] = m
        c.row_is_plan_a[r] = 1 if (len(row) > 0 and list(row[0]) == all_indices) else 0
    c.plan_a_only = 1 if conf.get("plan_a_masks") else 0
    return c


class Imputation(object):
    def __init__(self, net=None, config=None, count_by_prob=None, verbose=False):
        self.netGraph = net
        self.config = config
        self.verbose = verbose
        self.populations = list(config["pops"])
        self.loci = net.loci
        self.L = len(self.loci)
        self.P = len(self.populations)
        self.unk_priors = config["UNK_priors"]
        self.priority = config["priority"]
        if count_by_prob is None:
            self.count_by_prob = np.ones(self.P)
            if config.get("use_pops_count_file"):
                with open(config["pops_count_file"]) as f:
                    for i, line in enumerate(f):
                        self.count_by_prob[i] = float(line.strip().split(",")[2])
        else:
            self.count_by_prob = count_by_prob
        self.cfg = make_config(config, self.loci, self.P)
        # Plan_A_Matrix: typed-locus patterns that are matrix rows (impute.py:1592-1596 of the reference)
        self.type_allowed = None
        if config.get("plan_a_masks"):
            if getattr(net, "plan_a_masks", None) != config["plan_a_masks"]:
                raise ValueError("the Graph was not built for this Plan_A_Matrix")
            self.type_allowed = np.zeros(1 << self.L, dtype=np.uint8)
            self.type_allowed[config["plan_a_masks"]] = 1
        elif getattr(net, "plan_a_masks", None):
            raise ValueError("the Graph was built for a Plan_A_Matrix the configuration does not name")
        self.locus_index = {n: i for i, n in enumerate(self.loci)}
        self.batch_size = int(os.environ.get("GRIMB_BATCH", "65536"))
        self.workspaces = [int(x) for x in os.environ.get(
            "GRIMB_WORKSPACES", "%d,%d,%d" % (32 << 20, 512 << 20, 4 << 30)).split(",")]
        self._prior_index = {}
        self._priors = []
        self._backend = self._run_gpu
        # per-subject phase masks (bin_imputation_in_file; impute.py:2001-2005 of the reference)
        self.phase_masks = None
        bin_path = config.get("bin_imputation_input_file", "None")
        if bin_path and os.path.isfile(bin_path):
            import json
            with open(bin_path) as f:
                self.phase_masks = json.load(f)
        self._em_mr = False
        self.stats = {"subjects": 0, "pair_evals": 0, "plan": {0: 0, 1: 0, 2: 0, 3: 0}, "workspace_retries": 0}

    # ------------------------------------------------------------------ prior matrices
    def _prior_matrix(self, races1, races2):
        # same arithmetic, in the same order, as calc_priority_matrix (impute.py:1844-1924)
        pr = self.priority
        n = self.P
        M = np.zeros((n, n))
        eye = np.identity(n)
        for a in races1:
            for b in races2:
                if a == "" and b == "":
                    continue
                T = np.zeros((n, n))
                if a == "" or b == "":
                    r = self.populations.index(b) if a == "" else self.populations.index(a)
                    for i in range(n):
                        T[r, i] = T[r, i] + pr["gamma"] * 2
                    T = T + T.transpose()
                    T[r, r] -= pr["gamma"] * 2
                else:
                    r1 = self.populations.index(a)
                    r2 = self.populations.index(b)
                    for i in range(n):
                        T[r1, i] = T[r1, i] + pr["gamma"]
                        T[i, r2] = T[i, r2] + pr["gamma"]
                    T[r1, r2] -= pr["gamma"]
                    T[r1, r2] = T[r1, r2] + pr["alpha"]
                    if r1 != r2:
                        T = T + T.transpose()
                        T[r1, r1] -= pr["gamma"]
                        T[r2, r2] -= pr["gamma"]
                    T[r1, r1] += pr["delta"]
                    if r1 != r2:
                        T[r2, r2] += pr["delta"]
                T = pr["eta"] * np.ones((n, n)) + T + pr["beta"] * eye
                M += T
        total = 0
        for i in range(n):
            for j in range(n):
                M[i][j] = M[i][j] * self.count_by_prob[i] * self.count_by_prob[j]
                total += M[i][j]
        return M / total

    def _prior_for(self, race1, race2):
        """Index of the prior matrix for these race fields (impute.py:1956-1975)."""
        key = (race1, race2)
        idx = self._prior_index.get(key)
        if idx is not None:
            return idx
        n = self.P
        M = np.ones((n, n)) if self.unk_priors == "MR" else np.identity(n)
        if race1 or race2:
            known = False
            r1 = race1.split(";")
            for i, r in enumerate(r1):
                if r not in self.populations:
                    r1[i] = ""
                else:
                    known = True
            r2 = race2.split(";")
            for i, r in enumerate(r2):
                if r not in self.populations:
                    r2[i] = ""
                else:
                    known = True
            if known:
                M = self._prior_matrix(r1, r2)
        idx = len(self._priors)
        self._priors.append(np.ascontiguousarray(M, dtype=np.float64))
        self._prior_index[key] = idx
        return idx

    # ------------------------------------------------------------------ tokeniser
    def _encode_gl(self, gl):
        """GL string -> (class, typed_mask, counts [L][2], allele ids, unknown-name map).
        Mirrors clean_up_gl + gl2haps (impute.py:105-118,246-272)."""
        L = self.L
        gl = clean_up_gl(gl)
        if gl == "" or gl == " ":
            return H_PROBLEM, None
        t1, t2 = [], []
        for chunk in gl.split("^"):
            if chunk == "":
                return H_FAULT, None          # IndexError on chunk[0] in the reference
            if chunk[0] == "+":
                chunk = chunk[1:]
            sides = chunk.split("+")
            if len(sides) == 1:
                if sides == [""]:
                    continue
                return H_PROBLEM, None        # a locus without '+': gl2haps returns []
            t1.append(sides[0])
            t2.append(sides[1])
        if not t1:
            return H_FAULT, None              # 2 ** (0 - 1) phases: TypeError in the reference
        t1.sort()
        t2.sort()
        counts = np.zeros((L, 2), dtype=np.uint16)
        per_locus = [None] * L
        unknown = None
        ids_of = self.netGraph.allele_id
        n_tab = [len(a) for a in self.netGraph.alleles]
        cap = [(1 << b) - 1 for b in self.netGraph.key_bits]
        if self.type_allowed is not None:
            # input_type (impute.py:1574-1579): every typed locus is looked up first (KeyError -> raw line in
            # .problem); a pattern that is no matrix row -> comp_cand returns None -> .problem "i,id"
            pattern = []
            for a in t1:
                l = self.locus_index.get(a.split("/")[0].split("*")[0])
                if l is None:
                    return H_FAULT, None
                pattern.append(l)
            mask = 0
            for l in pattern:
                mask |= 1 << l
            if len(set(pattern)) != len(pattern) or not self.type_allowed[mask]:
                return H_PROBLEM, None
        for a, b in zip(t1, t2):
            la = a.split("/")
            lb = b.split("/")
            l = self.locus_index.get(la[0].split("*")[0])
            if l is None or per_locus[l] is not None:
                return (H_FAULT if self.config["planb"] else H_OK), "foreign"
            local = {}
            pair = []
            for lst in (la, lb):
                out = []
                for name in lst:
                    if name.split("*")[0] != self.loci[l]:
                        return (H_FAULT if self.config["planb"] else H_OK), "foreign"
                    i = ids_of[l].get(name)
                    if i is None:
                        i = local.get(name)
                        if i is None:
                            i = n_tab[l] + 1 + len(local)
                            if i > cap[l]:
                                return H_FAULT, None
                            local[name] = i
                    if i not in out:
                        out.append(i)
                pair.append(out)
            if local:
                if unknown is None:
                    unknown = {}
                for name, i in local.items():
                    unknown[(l, i)] = name
            per_locus[l] = pair
        mask = 0
        flat = []
        for l in range(L):
            if per_locus[l] is not None:
                mask |= 1 << l
                for x in range(2):
                    counts[l, x] = len(per_locus[l][x])
                    flat.extend(per_locus[l][x])
        return H_OK, (mask, counts, flat, unknown)

    # ------------------------------------------------------------------ batch execution
    def _run_gpu(self, cfg, batch, res, workspace):
        lib = self.netGraph.lib
        eng = self.netGraph.engine(workspace)
        return lib.grimb_impute_host(eng, C.byref(cfg), C.byref(batch), C.byref(res))

    def _run_batch(self, enc, workspace):
        """enc: list of (mask, counts, flat ids, prior index, phase mask).  -> _lib.ResultArrays of the call."""
        S, L = len(enc), self.L
        typed = np.zeros(S, np.uint16)
        counts = np.zeros((S, L, 2), np.uint16)
        off = np.zeros(S + 1, np.uint32)
        pri = np.zeros(S, np.uint32)
        pmask = np.zeros(S, np.uint16)
        flat = []
        for s, (mask, cn, ids, p, pm) in enumerate(enc):
            typed[s] = mask
            pmask[s] = pm
            if mask:
                counts[s] = cn
                flat.extend(ids)
            off[s + 1] = len(flat)
            pri[s] = p
        alle = np.array(flat if flat else [0], dtype=np.uint16)
        priors = np.ascontiguousarray(np.stack(self._priors)) if self._priors else np.ones((1, self.P, self.P))
        b = _lib.Batch()
        b.n_subjects = S
        b.typed_mask, b.counts, b.allele_off = typed.ctypes.data, counts.ctypes.data, off.ctypes.data
        b.alleles, b.n_alleles_total = alle.ctypes.data, int(off[S])
        b.prior_index, b.priors, b.n_priors = pri.ctypes.data, priors.ctypes.data, priors.shape[0]
        b.phase_mask = pmask.ctypes.data if self.phase_masks is not None else None
        words, general, hap, pop = self._result_caps(S, self._em_mr)
        res = _lib.ResultArrays(S, self.netGraph.kw, words=words, general=general, hap=hap, pop=pop)
        while True:
            t0 = time.perf_counter()
            rc = self._backend(self.cfg, b, res.struct, workspace)
            self.stats["abi_seconds"] = self.stats.get("abi_seconds", 0.0) + time.perf_counter() - t0
            if rc == _lib.E_CAPACITY:
                res.grow()
                continue
            if rc != 0:
                _lib.check(rc, "grimb_impute_host", self.netGraph.lib)
            break
        return res

    def _result_caps(self, S, em_mr):
        """First-attempt capacities of the result arrays of a batch of S subjects that may be ambiguous (words,
        general records, hap rows, pop rows): one general record per subject and the configured number of rows, so
        that such a batch rarely meets GRIMB_E_CAPACITY, which the library reports only after the kernels ran."""
        hap = max(1024, S * 2 * min(self.cfg.n_results, 16))
        pop = max(1024, S * 2 * min(self.cfg.n_pop_results, 4))
        if em_mr:
            pop += S * min(self.cfg.n_results, 16)   # the hap_pop_pair companion rows
        return [max(1024, S * 8), max(1024, S), hap, pop]

    # ------------------------------------------------------------------ formatting
    def _allele_name(self, l, i, unknown):
        al = self.netGraph.alleles[l]
        if 1 <= i <= len(al):
            return al[i - 1]
        return unknown[(l, i)]

    def _decode(self, key, unknown):
        g = self.netGraph
        key = int(key) if g.kw == 1 else int(key[0]) | (int(key[1]) << 64)
        out = []
        for l in range(self.L):
            i = (key >> g.shift[l]) & ((1 << g.key_bits[l]) - 1)
            if i:
                out.append(self._allele_name(l, i, unknown))
            else:
                out.append(None)
        return out

    def _pop_name(self, p):
        return "all_pops" if p == _lib.ALL_POPS else self.populations[p]

    def _subject_rows(self, res, k, ids, unknown):
        """Result of subject k of one ABI call as plain Python rows (include/grimb200.h, ABI v4):
        -> dict(status, plan_umug, plan_pmug, tot_umug, tot_pmug, evals, umug [(loci pairs, prob)],
        umug_pops / pmug_pops [(pop a, pop b, prob)], pmug [(hap 1 names, hap 2 names, prob)],
        pmug_pairs [(pop a, pop b)] (the hap_pop_pair companions))."""
        c = res.compact[k]
        kf = int(c["kind_flags"])
        kind, has, n_pmug = kf & 3, bool(kf & _lib.KIND_HAS_RESULTS), kf >> 4
        out = {"status": int(c["status"]), "umug": [], "umug_pops": [], "pmug": [], "pmug_pops": [], "pmug_pairs": []}
        if kind == _lib.KIND_GENERAL:
            if int(c["off"]) == _lib.NO_RECORD:
                out.update(plan_umug=0, plan_pmug=0, tot_umug=0, tot_pmug=0)
                return out
            r = res.general[int(c["off"])]
            ho, po = int(r["hap_off"]), int(r["pop_off"])
            nu, np_, nup, npp = (int(r[f]) for f in ("n_umug", "n_pmug", "n_umug_pops", "n_pmug_pops"))
            out.update(plan_umug=int(r["plan_umug"]), plan_pmug=int(r["plan_pmug"]), tot_umug=int(r["tot_umug"]),
                       tot_pmug=int(r["tot_pmug"]))
            hr, pr = res.hap_rows, res.pop_rows
            for q in range(nu):
                row = hr[ho + q]
                a, b = self._decode(row["a"], unknown), self._decode(row["b"], unknown)
                out["umug"].append(([(x, y) for x, y in zip(a, b) if x is not None], float(row["prob"])))
            for q in range(np_):
                row = hr[ho + nu + q]
                out["pmug"].append(([x for x in self._decode(row["a"], unknown) if x is not None],
                                    [x for x in self._decode(row["b"], unknown) if x is not None], float(row["prob"])))
                if self._em_mr:
                    pp = pr[po + nup + npp + q]
                    out["pmug_pairs"].append((self._pop_name(int(pp["pa"])), self._pop_name(int(pp["pb"]))))
            for q in range(nup):
                row = pr[po + q]
                out["umug_pops"].append((self._pop_name(int(row["pa"])), self._pop_name(int(row["pb"])), float(row["prob"])))
            for q in range(npp):
                row = pr[po + nup + q]
                out["pmug_pops"].append((self._pop_name(int(row["pa"])), self._pop_name(int(row["pb"])), float(row["prob"])))
            return out
        # SIMPLE / TYPED: every locus typed, one allele per side; rows follow from the subject's own alleles
        L = self.L
        names = [(self._allele_name(l, ids[2 * l], unknown), self._allele_name(l, ids[2 * l + 1], unknown)) for l in range(L)]
        total, off = float(c["total"]), int(c["off"])
        w = res.words
        cfg = self.cfg
        if kind == _lib.KIND_SIMPLE and n_pmug == 15:
            # long form (more than four PMUG rows): a count word, a word of phase ids, then the probabilities
            n_pmug = min(16, int(w[off]))
            phases = [(int(w[off + 1]) >> (4 * q)) & 15 for q in range(n_pmug)]
            probs = [float(x) for x in w[off + 2:off + 2 + n_pmug].view(np.float64)]
            pops = [(self.populations[0], self.populations[0], total)] if (has and cfg.n_pop_results >= 1) else []
        elif kind == _lib.KIND_SIMPLE:
            phases = [(int(c["phases"]) >> (4 * q)) & 15 for q in range(n_pmug)]
            probs = [float(w[off + q:off + q + 1].view(np.float64)[0]) for q in range(n_pmug)] if kf & _lib.KIND_WORDS \
                else [total] * n_pmug
            pops = [(self.populations[0], self.populations[0], total)] if (has and cfg.n_pop_results >= 1) else []
        else:
            hdr = int(w[off])
            n_pops = hdr & 0xFFFF
            phases = [(hdr >> (16 + 12 * q)) & 0xFFF for q in range(n_pmug)]
            probs = [float(x) for x in w[off + 1:off + 1 + n_pmug].view(np.float64)]
            pp = w[off + 1 + n_pmug:off + 1 + n_pmug + n_pops].view(np.float64)
            codes = w[off + 1 + n_pmug + n_pops:off + 1 + n_pmug + n_pops + (n_pops + 3) // 4].view(np.uint16)
            pops = [(self.populations[int(codes[q]) >> 8], self.populations[int(codes[q]) & 0xFF], float(pp[q]))
                    for q in range(n_pops)]
        out.update(plan_umug=_lib.PLAN_A if cfg.output_umug else 0, plan_pmug=_lib.PLAN_A if cfg.output_pmug else 0,
                   tot_umug=1 if (has and cfg.output_umug) else 0, tot_pmug=(max(1, n_pmug) if has else 0) if cfg.output_pmug else 0)
        if cfg.output_pmug:
            for ph, pr_ in zip(phases, probs):
                out["pmug"].append(([names[l][(ph >> l) & 1] for l in range(L)],
                                    [names[l][1 - ((ph >> l) & 1)] for l in range(L)], pr_))
            out["pmug_pops"] = list(pops)
        if cfg.output_umug and has:
            if cfg.n_results >= 1:
                out["umug"].append((list(names), total))
            out["umug_pops"] = list(pops)
        return out

    def _format_subject(self, sid, rows, files):
        cfgd = self.config
        if cfgd["output_haplotypes"]:
            dst = files["pmug"]
            for k, (h1, h2, prob) in enumerate(rows["pmug"]):
                if self._em_mr:
                    # write_best_hap_race_pairs (impute.py:79-99): "hap;pop,hap;pop"
                    pa, pb = rows["pmug_pairs"][k]
                    dst.append(sid + "," + "~".join(h1) + ";" + pa + "," + "~".join(h2) + ";" + pb + "," + str(prob)
                               + "," + str(k) + "\n")
                    continue
                dst.append(sid + "," + "~".join(h1) + "+" + "~".join(h2) + "," + str(prob) + "," + str(k) + "\n")
            dst = files["pmug_pops"]
            for k, (pa, pb, prob) in enumerate(rows["pmug_pops"]):
                dst.append(sid + "," + pa + "," + pb + "," + str(prob) + "," + str(k) + "\n")
        if cfgd["output_MUUG"]:
            dst = files["umug"]
            for k, (pairs, prob) in enumerate(rows["umug"]):
                geno = "^".join("+".join(sorted([x, y])) for x, y in pairs)
                dst.append(sid + "," + geno + "," + str(prob) + "," + str(k) + "\n")
            dst = files["umug_pops"]
            planc = rows["plan_umug"] == _lib.PLAN_C
            for k, (pa, pb, prob) in enumerate(rows["umug_pops"]):
                names = sorted([pa, pb])
                text = str(prob)
                if planc and rows["tot_umug"] == 0:
                    text = "0"  # sum() of an empty dict is the int 0 (impute.py:1376)
                dst.append(sid + "," + names[0] + "," + names[1] + "," + text + "," + str(k) + "\n")

    # ------------------------------------------------------------------ public entry points
    def impute_lines(self, lines, first_index=0, em_mr=False, em=False):
        """Imputes an iterable of input lines; returns the six output texts as lists of rows.
        em_mr: the hap_pop_pair output mode of grim.grim.impute (impute.py:2079-2088); em: no Plan C for
        the haplotype output (impute.py:1648)."""
        self._em_mr = bool(em_mr)
        self.cfg.hap_pop_pair = 1 if em_mr else 0
        self.cfg.em = 1 if em else 0
        files = {k: [] for k in ("umug", "umug_pops", "pmug", "pmug_pops", "miss", "problem")}
        pending = []
        for i, raw in enumerate(lines, first_index):
            pending.append((i, raw))
            if len(pending) >= self.batch_size:
                self._process(pending, files)
                pending = []
        if pending:
            self._process(pending, files)
        return files

    def impute_one(self, subject_id, gl, binary, race1, race2, priority, epsilon, n, MUUG_output, haps_output, planb, em):
        """The per-subject seam of the reference (impute.py:1940-1983; consumer scripts/parallel-imputation.py):
        -> (subject_id, res_muugs, res_haps) with the reference's structures --
            res_muugs = {"MaxProb", "Haps": {genotype: prob}, "Pops": {"pop,pop": prob}}   (dicts in insertion order)
            res_haps  = {"MaxProb", "Haps": [[hap1, hap2]], "Probs": [prob], "Pops": [[pop1, pop2]]}   (un-merged)
        or (subject_id, None, None) where comp_cand gives up.  A compatibility mode: one subject per call through
        the general kernel with GrimbConfig.encounter_order (rows in traversal order, nothing ranked) and
        hap_pop_pair (the accepted pairs, un-merged); the batch entry points are the fast path.  `n` is accepted
        and unused, as in the reference.  MaxProb is the largest single-pair probability of the haplotype-pair
        evaluation (the genotype evaluation meets the same pairs whenever both end in the same plan)."""
        saved = (self.cfg.epsilon, self.cfg.planb, self.cfg.em, self.cfg.hap_pop_pair, self.cfg.encounter_order,
                 self.cfg.output_umug, self.cfg.output_pmug, self.cfg.n_results, self.cfg.n_pop_results, self._em_mr,
                 self.priority, self._prior_index, self._priors)
        limit = int(os.environ.get("GRIMB_IMPUTE_ONE_ROWS", "200000"))
        try:
            self.cfg.epsilon = float(epsilon)
            self.cfg.planb = 1 if planb else 0
            self.cfg.em = 1 if em else 0
            self.cfg.hap_pop_pair, self.cfg.encounter_order = 1, 1
            self.cfg.output_umug, self.cfg.output_pmug = 1, 1
            self.cfg.n_results = self.cfg.n_pop_results = limit
            self._em_mr = True
            if priority is not None and priority != self.priority:
                self.priority, self._prior_index, self._priors = priority, {}, []
            default_muugs = {"MaxProb": 0, "Haps": {}, "Pops": {}}
            default_haps = {"Haps": "Nan", "Probs": 0, "Pops": {}}
            pidx = self._prior_for(race1, race2)
            if not gl:
                return subject_id, None, None
            hclass, payload = self._encode_gl(gl)
            if hclass == H_PROBLEM:
                return subject_id, None, None
            if hclass == H_FAULT:
                raise RuntimeError("the reference raises inside this subject")
            if payload == "foreign":       # nothing is imputed (Plan B off): the defaults come back
                return subject_id, default_muugs, default_haps
            mask, counts, flat, unknown = payload
            pm = 0xFFFF
            if binary is not None:
                pm = _phase_mask(binary)
            had_masks = self.phase_masks
            if binary is not None and had_masks is None:
                self.phase_masks = {}      # makes _run_batch hand the mask array to the kernels
            try:
                rows = None
                for tier in self.workspaces:
                    out = self._run_batch([(mask, counts, flat, pidx, pm)], tier)
                    if out.compact["status"][0] != _lib.ST_WORKSPACE:
                        rows = self._subject_rows(out, 0, flat, unknown)
                        break
                if rows is None:
                    raise MemoryError("the subject exceeds the largest workspace tier (GRIMB_WORKSPACES)")
            finally:
                self.phase_masks = had_masks
            if rows["status"] == _lib.ST_FAULT:
                raise RuntimeError("the reference raises inside this subject")
            if rows["status"] == _lib.ST_NO_PHASES:
                return subject_id, default_muugs, default_haps
            if rows["tot_pmug"] > limit or rows["tot_umug"] > limit:
                raise MemoryError("more than GRIMB_IMPUTE_ONE_ROWS = %d result rows" % limit)
            max_prob = max([p for _a, _b, p in rows["pmug"]], default=0)
            res_muugs, res_haps = default_muugs, default_haps
            if MUUG_output:
                res_muugs = {"MaxProb": max_prob, "Haps": {}, "Pops": {}}
                for pairs, prob in rows["umug"]:
                    res_muugs["Haps"]["^".join("+".join(sorted([x, y])) for x, y in pairs)] = prob
                for pa, pb, prob in rows["umug_pops"]:
                    res_muugs["Pops"][",".join(sorted([pa, pb]))] = prob
            if haps_output:
                res_haps = {"MaxProb": max_prob, "Haps": [], "Probs": [], "Pops": []}
                for (h1, h2, prob), (pa, pb) in zip(rows["pmug"], rows["pmug_pairs"]):
                    res_haps["Haps"].append(["~".join(h1), "~".join(h2)])
                    res_haps["Probs"].append(prob)
                    res_haps["Pops"].append([pa, pb])
            return subject_id, res_muugs, res_haps
        finally:
            (self.cfg.epsilon, self.cfg.planb, self.cfg.em, self.cfg.hap_pop_pair, self.cfg.encounter_order,
             self.cfg.output_umug, self.cfg.output_pmug, self.cfg.n_results, self.cfg.n_pop_results, self._em_mr,
             self.priority, self._prior_index, self._priors) = saved

    def _process(self, pending, files):
        cfgd = self.config
        meta = []   # (line index, id, raw, host class, unknown map)
        enc = []
        for i, raw in pending:
            raw = raw.rstrip()
            fields = raw.split(",") if "," in raw else raw.split("%")
            sid = fields[0]
            hclass, unknown, item = H_OK, None, (0, None, None, 0, 0xFFFF)
            pm = 0xFFFF
            if self.phase_masks is not None and len(fields) >= 2:
                bits = self.phase_masks.get(sid)
                if bits is None:
                    hclass = H_FAULT                   # KeyError f_bin[subject_id] -> raw line in .problem
                else:
                    pm = _phase_mask(bits)
            if len(fields) < 2 or len(fields) == 3 or hclass == H_FAULT:
                hclass = H_FAULT                       # IndexError in the reference's line parser
            else:
                gl = fields[1]
                race1 = race2 = None
                if len(fields) > 2:
                    race1, race2 = fields[2], fields[3]
                pidx = self._prior_for(race1, race2)
                if not gl:
                    hclass = H_PROBLEM
                else:
                    hclass, payload = self._encode_gl(gl)
                    if hclass == H_OK and payload != "foreign":
                        mask, counts, flat, unknown = payload
                        item = (mask, counts, flat, pidx, pm)
            meta.append((i, sid, raw, hclass, unknown))
            enc.append(item)
        # per-CTA workspace tiers: subjects that overflow one tier are re-issued on the next
        where = {}
        todo = list(range(len(enc)))
        for tier in self.workspaces:
            out = self._run_batch([enc[s] for s in todo], tier)
            self.stats["pair_evals"] += int(out.totals[4])
            again = []
            for k, s in enumerate(todo):
                if out.compact["status"][k] == _lib.ST_WORKSPACE:
                    again.append(s)
                else:
                    where[s] = (out, k)
            if not again:
                break
            self.stats["workspace_retries"] += len(again)
            todo = again
        else:
            raise MemoryError("a subject exceeds the largest workspace tier (GRIMB_WORKSPACES)")
        for s, (i, sid, raw, hclass, unknown) in enumerate(meta):
            self.stats["subjects"] += 1
            if hclass == H_PROBLEM:
                files["problem"].append(str(i) + "," + str(sid) + "\n")
                continue
            if hclass == H_FAULT:
                files["problem"].append(raw + "\n")
                continue
            r, k = where[s]
            rows = self._subject_rows(r, k, enc[s][2], unknown)
            st = rows["status"]
            if st == _lib.ST_FAULT:
                files["problem"].append(raw + "\n")
                continue
            if st == _lib.ST_NO_PHASES:
                # nothing opens (reference: defaults returned, the PMUG writer then raises)
                if cfgd["output_haplotypes"]:
                    files["problem"].append(raw + "\n")
                continue
            tot_u, tot_p = rows["tot_umug"], rows["tot_pmug"]
            self.stats["plan"][rows["plan_umug"] if cfgd["output_MUUG"] else rows["plan_pmug"]] += 1
            pm_empty = (tot_p == 0) if cfgd["output_haplotypes"] else False
            if self.cfg.plan_a_only and self.cfg.planb and (
                    (cfgd["output_MUUG"] and tot_u == 0) or (cfgd["output_haplotypes"] and tot_p == 0)):
                raise NotImplementedError(
                    "subject %s (line %d) leaves Plan A without a result under a Plan_A_Matrix: the reference's "
                    "Plan B is not well defined there; set \"planb\": false to write such subjects to the .miss file"
                    % (sid, i))
            if pm_empty and tot_u == 0:
                files["miss"].append(str(i) + "," + str(sid) + "\n")
            self._format_subject(sid, rows, files)

    # ------------------------------------------------------------------ device-resident genotype interface
    def prior_index(self, race1, race2):
        """Index of the prior matrix for the race fields (race1, race2) of an input line (impute.py:1956-1975 of
        the reference), for the prior_index argument of impute_genotypes."""
        return self._prior_for(race1, race2)

    def encode_genotypes(self, gl_strings):
        """GL strings -> (ids uint16 [S][L][2] for impute_genotypes, unknown-name maps, text-path line indices).
        ids[s, l] = the (side 0, side 1) allele ids of locus l (0/0: untyped); unknown[s] maps (locus, id) to the
        name of an allele absent from the table, or is None.  A line with allele ambiguity, or one the tokeniser
        classes as a problem or a fault, gets an all-zero row (it comes back SKIPPED) and its index is listed in
        the third value: such lines belong on the text path (impute_text)."""
        S, L = len(gl_strings), self.L
        ids = np.zeros((S, L, 2), np.uint16)
        unknown = [None] * S
        text_path = []
        for s, gl in enumerate(gl_strings):
            hclass, payload = self._encode_gl(gl) if gl else (H_PROBLEM, None)
            if hclass != H_OK or payload == "foreign" or (payload[1] > 1).any():
                text_path.append(s)
                continue
            mask, _counts, flat, unknown[s] = payload
            k = 0
            for l in range(L):
                if (mask >> l) & 1:
                    ids[s, l] = flat[k:k + 2]
                    k += 2
        return ids, unknown, text_path

    def encode_genotype_lists(self, gl_strings):
        """GL strings -> (counts uint16 [S][L][2], alleles uint16 [N], unknown-name maps, text-path line indices) for
        impute_genotype_lists.  counts[s, l, x] = the number of ids listed on side x of locus l (0/0: untyped);
        alleles = the ids concatenated subject-major, locus ascending, side 0 then side 1, each list in the order it
        was written with repeats dropped; unknown[s] as in encode_genotypes.  A line the tokeniser classes as a
        problem or a fault, or one naming a locus foreign to the table, gets zero counts (it comes back SKIPPED) and
        its index is listed in the fourth value: such lines belong on the text path (impute_text)."""
        S, L = len(gl_strings), self.L
        counts = np.zeros((S, L, 2), np.uint16)
        unknown = [None] * S
        text_path = []
        flat = []
        for s, gl in enumerate(gl_strings):
            hclass, payload = self._encode_gl(gl) if gl else (H_PROBLEM, None)
            if hclass != H_OK or payload == "foreign":
                text_path.append(s)
                continue
            _mask, counts[s], ids, unknown[s] = payload
            flat.extend(ids)
        return counts, np.array(flat, np.uint16), unknown, text_path

    def phase_masks_for(self, subject_ids):
        """Phase masks of the configured bin_imputation_in_file for these subject ids, built as impute_lines builds
        them: -> (uint16 [S] for the phase_mask argument of impute_genotype_lists, indices of the ids the file has
        no entry for).  Those subjects get 0xFFFF here; the text path faults their lines (raw line in .problem)."""
        if self.phase_masks is None:
            raise ValueError("no bin_imputation_in_file is configured")
        masks = np.full(len(subject_ids), 0xFFFF, np.uint16)
        missing = []
        for s, sid in enumerate(subject_ids):
            bits = self.phase_masks.get(sid)
            if bits is None:
                missing.append(s)
            else:
                masks[s] = _phase_mask(bits)
        return masks, missing

    def _check_genotype_modes(self, em_mr, em):
        if em_mr or self.cfg.hap_pop_pair:
            raise NotImplementedError("impute_genotypes: the hap_pop_pair / em_mr output mode takes impute_genotype_lists")
        if em or self.cfg.em:
            raise NotImplementedError("impute_genotypes: the em mode takes impute_genotype_lists")
        if self.cfg.encounter_order:
            raise NotImplementedError("impute_genotypes: encounter_order (the impute_one seam) stays on impute_one")
        if self.phase_masks is not None:
            raise NotImplementedError("impute_genotypes: bin_imputation_in_file phase masks take impute_genotype_lists")

    @staticmethod
    def _device_int16(x, dev, what):
        """numpy array or CUDA tensor on `dev` -> contiguous CUDA int16 tensor with the same 16-bit patterns."""
        import torch
        if isinstance(x, torch.Tensor):
            if not x.is_cuda or x.device != dev:
                raise ValueError("%s must be a numpy array or a CUDA tensor on the table's device (%s)" % (what, dev))
            t = x
        else:
            t = torch.from_numpy(np.ascontiguousarray(x))
        t = t.view(torch.int16) if t.dtype in (torch.uint16, torch.int16) else t.to(torch.int32).to(torch.int16)
        return t.to(dev).contiguous()

    def impute_genotypes(self, ids, prior_index=None, em_mr=False, em=False):
        """Imputes a batch of typed genotypes on the device: ids [S][L][2] allele ids as encode_genotypes returns
        them (Graph.allele_id; 0/0 = untyped locus; ids past the table = subject-local unknown alleles), prior_index
        [S] optional (Imputation.prior_index).  The batch is encoded, imputed and decoded on the GPU
        (grimb_batch_from_genotypes, the imputation kernels, grimb_results_rows).  A CUDA torch tensor on the
        table's device stays there and the results are CUDA tensors; a numpy array gives numpy results.
        -> GenotypeResults.  Subjects that overflow a workspace tier are re-issued on the next one.  Ambiguous
        genotypes, phase masks and the EM modes take impute_genotype_lists."""
        import torch
        self._check_genotype_modes(em_mr, em)
        g = self.netGraph
        dev = torch.device("cuda", g.device)
        as_numpy = not isinstance(ids, torch.Tensor)
        t = self._device_int16(ids, dev, "ids")
        if t.dim() != 3 or t.shape[1] != self.L or t.shape[2] != 2:
            raise ValueError("ids must be [S][%d][2]" % self.L)
        ta = self.type_allowed.ctypes.data if self.type_allowed is not None else None
        self.cfg.hap_pop_pair = self.cfg.em = 0

        def encoder(todo):
            sub = t if todo is None else t.index_select(0, todo).contiguous()
            n = int(sub.shape[0])

            def encode(eng, pri, priors, b, sp):
                _lib.check(g.lib.grimb_batch_from_genotypes(eng, sub.data_ptr(), n, pri, priors.data_ptr(), priors.shape[0],
                                                            ta, C.byref(b), sp), "grimb_batch_from_genotypes", g.lib)
            return n, encode
        # typed subjects are mostly SIMPLE / TYPED records: few general records and hap rows
        caps = lambda n: [n * 2 + 1024, n // 8 + 1024, n // 4 + 1024, n // 4 + 1024]
        return self._impute_device(encoder, int(t.shape[0]), prior_index, dev, as_numpy, caps)

    def impute_genotype_lists(self, counts, alleles, prior_index=None, phase_mask=None, em_mr=False, em=False):
        """Imputes a batch of genotypes with allele ambiguity on the device: counts [S][L][2] and alleles [N] as
        encode_genotype_lists returns them (a side's list repeating an id is fine: the repeat is dropped),
        prior_index [S] optional (Imputation.prior_index), phase_mask [S] optional (uint16, bit m = the m-th typed
        locus may switch sides; Imputation.phase_masks_for builds it from the configured bin_imputation_in_file,
        and then it is required).  em_mr: the hap_pop_pair output mode (GenotypeResults.pmug_pairs gets each PMUG
        row's two populations); em: no Plan C for the haplotype output; both for this call only.  The batch is
        encoded (grimb_batch_from_genotype_lists), imputed and decoded on the GPU.  CUDA tensors on the table's
        device stay there and the results are CUDA tensors; numpy counts give numpy results.  -> GenotypeResults.
        The counts must list N ids in all (ValueError / RuntimeError otherwise).  Subjects that overflow a
        workspace tier are re-issued on the next one."""
        import torch
        if self.cfg.encounter_order:
            raise NotImplementedError("impute_genotype_lists: encounter_order (the impute_one seam) stays on impute_one")
        if self.phase_masks is not None and phase_mask is None:
            raise ValueError("bin_imputation_in_file is configured: pass phase_mask (Imputation.phase_masks_for)")
        g = self.netGraph
        dev = torch.device("cuda", g.device)
        as_numpy = not isinstance(counts, torch.Tensor)
        c = self._device_int16(counts, dev, "counts")
        a = self._device_int16(alleles, dev, "alleles")
        if c.dim() != 3 or c.shape[1] != self.L or c.shape[2] != 2:
            raise ValueError("counts must be [S][%d][2]" % self.L)
        if a.dim() != 1:
            raise ValueError("alleles must be one-dimensional")
        S = int(c.shape[0])
        pm = None
        if phase_mask is not None:
            pm = self._device_int16(phase_mask, dev, "phase_mask")
            if tuple(pm.shape) != (S,):
                raise ValueError("phase_mask must be [S]")
        ta = self.type_allowed.ctypes.data if self.type_allowed is not None else None

        def encoder(todo):
            sc, sa, spm = c, a, pm
            if todo is not None:
                # the re-issued subjects' lists, gathered from their input offsets
                n_in = (c.to(torch.int32) & 0xFFFF).sum((1, 2)).to(torch.int64)
                in_off = torch.cumsum(n_in, 0) - n_in
                cnt = n_in.index_select(0, todo)
                total = int(cnt.sum())
                owner = torch.repeat_interleave(torch.arange(todo.numel(), device=dev), cnt, output_size=total)
                first = torch.cumsum(cnt, 0) - cnt
                src = in_off.index_select(0, todo)[owner] + torch.arange(total, device=dev) - first[owner]
                sc, sa = c.index_select(0, todo).contiguous(), a.index_select(0, src).contiguous()
                spm = pm.index_select(0, todo).contiguous() if pm is not None else None
            n = int(sc.shape[0])

            def encode(eng, pri, priors, b, sp):
                _lib.check(g.lib.grimb_batch_from_genotype_lists(
                    eng, sc.data_ptr(), sa.data_ptr(), int(sa.numel()), n, pri, priors.data_ptr(), priors.shape[0],
                    spm.data_ptr() if spm is not None else None, ta, C.byref(b), sp), "grimb_batch_from_genotype_lists", g.lib)
            return n, encode
        saved = (self.cfg.hap_pop_pair, self.cfg.em)
        self.cfg.hap_pop_pair, self.cfg.em = (1 if em_mr else 0), (1 if em else 0)
        try:
            return self._impute_device(encoder, S, prior_index, dev, as_numpy,
                                       lambda n: self._result_caps(n, bool(em_mr)))
        finally:
            self.cfg.hap_pop_pair, self.cfg.em = saved

    def _impute_device(self, encoder, S, prior_index, dev, as_numpy, result_caps):
        """The tier loop of impute_genotypes / impute_genotype_lists.  encoder(todo) -> (n, encode) for the subjects
        `todo` (CUDA int64 indices; None = the whole batch), where encode(engine, prior_index pointer, priors, batch,
        stream) builds their batch on the device; result_caps(n) -> the first-attempt capacities of their result
        arrays (words, general records, hap rows, pop rows)."""
        import torch
        g = self.netGraph
        pidx = self._prior_for(None, None)   # the matrix of a line without race fields (and priors never empty)
        if prior_index is None:
            pri = None if pidx == 0 else torch.full((S,), pidx, dtype=torch.int32, device=dev)
        else:
            pri = torch.as_tensor(np.asarray(prior_index) if not isinstance(prior_index, torch.Tensor) else prior_index)
            if pri.shape != (S,) or (S and (int(pri.min()) < 0 or int(pri.max()) >= len(self._priors))):
                raise ValueError("prior_index must be [S] indices from Imputation.prior_index")
            pri = pri.to(device=dev, dtype=torch.int32).contiguous()
        priors = torch.from_numpy(np.ascontiguousarray(np.stack(self._priors))).to(dev)
        stream = torch.cuda.current_stream(dev)
        out = None
        todo = None   # indices of the subjects re-issued on this tier (None: the whole batch)
        retries = reruns = 0
        for tier in self.workspaces:
            n, encode = encoder(todo)
            sub_pri = pri if (pri is None or todo is None) else pri.index_select(0, todo).contiguous()
            part = self._genotype_pass(encode, n, sub_pri, priors, tier, stream, result_caps(n))
            reruns += part.pop("capacity_reruns")
            out = part if todo is None else _splice_rows(out, part, todo)
            again = (part["status"] == _lib.ST_WORKSPACE).nonzero().flatten()
            if again.numel() == 0:
                break
            todo = again if todo is None else todo.index_select(0, again)
            retries += int(again.numel())
        else:
            raise MemoryError("a subject exceeds the largest workspace tier (GRIMB_WORKSPACES)")
        self.stats["workspace_retries"] += retries
        self.stats["subjects"] += S
        if self.cfg.plan_a_only and self.cfg.planb and S:
            st = out["status"] == _lib.ST_OK
            left = st & (((out["tot_umug"] == 0) & bool(self.cfg.output_umug)) | ((out["tot_pmug"] == 0) & bool(self.cfg.output_pmug)))
            if bool(left.any()):
                s = int(left.nonzero()[0, 0])
                raise NotImplementedError(
                    "subject %d leaves Plan A without a result under a Plan_A_Matrix: the reference's Plan B is not "
                    "well defined there; set \"planb\": false to write such subjects to the .miss file" % s)
        out["capacity_reruns"] = reruns
        return GenotypeResults(out, g.alleles, self.populations, retries, as_numpy)

    def _genotype_pass(self, encode, S, pri, priors, tier, stream, caps):
        """One tier: encode (see _impute_device), impute and decode S subjects -> dict of CUDA tensors, and the
        number of times grimb_impute_device ran again on larger result arrays ("capacity_reruns")."""
        import torch
        g, lib = self.netGraph, self.netGraph.lib
        dev = priors.device
        eng = g.engine(tier)
        L = self.L
        sp = C.c_void_p(stream.cuda_stream)
        b = _lib.Batch()
        encode(eng, pri.data_ptr() if pri is not None else None, priors, b, sp)
        hap_sz = 24 if g.kw == 1 else 40
        totals = np.zeros(9, np.int64)
        reruns = 0
        while True:
            compact = torch.empty(max(1, S) * 16, dtype=torch.uint8, device=dev)
            bufs = [torch.empty(c * sz, dtype=torch.uint8, device=dev) for c, sz in zip(caps, (8, 48, hap_sz, 16))]
            r = _lib.Results()
            r.compact, r.totals = compact.data_ptr(), totals.ctypes.data
            r.words, r.word_capacity = bufs[0].data_ptr(), caps[0]
            r.general, r.general_capacity = bufs[1].data_ptr(), caps[1]
            r.hap_rows, r.hap_capacity = bufs[2].data_ptr(), caps[2]
            r.pop_rows, r.pop_capacity = bufs[3].data_ptr(), caps[3]
            rc = lib.grimb_impute_device(eng, C.byref(self.cfg), C.byref(b), C.byref(r), sp)
            if rc == _lib.E_CAPACITY:
                caps = [max(c, int(x)) for c, x in zip(caps, totals[:4])]
                reruns += 1
                continue
            _lib.check(rc, "grimb_impute_device", lib)
            break
        out = {"status": torch.empty(S, dtype=torch.uint8, device=dev), "plan_umug": torch.empty(S, dtype=torch.uint8, device=dev),
               "plan_pmug": torch.empty(S, dtype=torch.uint8, device=dev), "flags": torch.empty(S, dtype=torch.uint8, device=dev),
               "tot_umug": torch.empty(S, dtype=torch.int32, device=dev), "tot_pmug": torch.empty(S, dtype=torch.int32, device=dev),
               "pair_evals": int(totals[4]), "capacity_reruns": reruns}
        for k in _lib.ROW_KINDS:
            out[k + "_off"] = torch.empty(S + 1, dtype=torch.int64, device=dev)
        width = (2 * L, 2 * L, 2, 2)
        rcap = list(getattr(self, "_row_caps", (S + 1024, 2 * S + 1024, S + 1024, S + 1024)))
        rtot = np.zeros(4, np.int64)
        pairs = bool(self.cfg.hap_pop_pair)
        while True:
            rows = _lib.Rows()
            if pairs:
                out["pmug_pairs"] = torch.empty((rcap[1], 2), dtype=torch.int16, device=dev)
                rows.pmug_pairs = out["pmug_pairs"].data_ptr()
            for f in ("status", "plan_umug", "plan_pmug", "flags", "tot_umug", "tot_pmug"):
                setattr(rows, f, out[f].data_ptr())
            for i, k in enumerate(_lib.ROW_KINDS):
                out[k] = torch.empty((rcap[i], width[i]), dtype=torch.int16, device=dev)
                out[k + "_prob"] = torch.empty(rcap[i], dtype=torch.float64, device=dev)
                rows.off[i], rows.rows[i], rows.prob[i] = out[k + "_off"].data_ptr(), out[k].data_ptr(), out[k + "_prob"].data_ptr()
                rows.capacity[i] = rcap[i]
            rows.totals = rtot.ctypes.data
            rc = lib.grimb_results_rows(eng, C.byref(self.cfg), C.byref(b), C.byref(r), C.byref(rows), sp)
            if rc == _lib.E_CAPACITY:
                rcap = [max(c, int(x)) for c, x in zip(rcap, rtot)]
                continue
            _lib.check(rc, "grimb_results_rows", lib)
            break
        shapes = ((L, 2), (2, L), (2,), (2,))
        for i, k in enumerate(_lib.ROW_KINDS):
            out[k] = out[k][:int(rtot[i])].reshape((int(rtot[i]),) + shapes[i])
            out[k + "_prob"] = out[k + "_prob"][:int(rtot[i])]
        if pairs:
            out["pmug_pairs"] = out["pmug_pairs"][:int(rtot[1])]
        return out

    # ------------------------------------------------------------------ EM helpers (host only)
    # open_gl_string / open_phases_for_em (impute.py:305-351 of the reference) are list-building
    # utilities the EM driver calls around imputation; they involve no frequency lookup, so they are
    # plain host code here as well.  Same return structure: [[ [opened haplotypes of side 1] ],
    # [ [opened haplotypes of side 2] ]] per phase, each haplotype a list of allele names.
    @staticmethod
    def _gl2haps_names(gl_string):
        if gl_string == "" or gl_string == " ":
            return []
        t1, t2, n = [], [], 0
        for chunk in gl_string.split("^"):
            if chunk[0] == "+":
                chunk = chunk[1:]
            cur = chunk.split("+")
            if len(cur) == 1:
                if cur == [""]:
                    continue
                return []
            t1.append(cur[0])
            t2.append(cur[1])
            n += 1
        return {"Genotype": [sorted(t1), sorted(t2)], "N_Loc": n}

    @staticmethod
    def gen_phases(gen, n_loci, b_phases=None):
        """Host restatement of the phase enumeration the kernels perform (names instead of ids)."""
        allowed = None if b_phases is None else {i for i, e in enumerate(b_phases) if e == 1}
        out, seen = [], set()
        for i in range(2 ** (n_loci - 1)):
            pick = [(i >> m) & 1 if (allowed is None or m in allowed) else 0 for m in range(n_loci)]
            h1 = [gen[pick[k]][k] for k in range(n_loci)]
            h2 = [gen[1 - pick[k]][k] for k in range(n_loci)]
            a, b = "~".join(h1) + "^" + "~".join(h2), "~".join(h2) + "^" + "~".join(h1)
            if a not in seen or b not in seen:
                seen.add(a)
                seen.add(b)
                out.append([h1, h2])
        return out

    def open_gl_string(self, gl_string, cutoff):
        chrom = self._gl2haps_names(gl_string)
        if chrom == []:
            return None
        phases = self.gen_phases(chrom["Genotype"], chrom["N_Loc"], None)
        if phases == []:
            return None
        return self.open_phases_for_em(phases, chrom["N_Loc"], cutoff)

    def open_phases_for_em(self, haps, N_Loc, cutoff):
        import itertools
        phases = []
        for pair in haps:
            sides = []
            for k in range(2):
                splits = [tuple(a.split("/")) for a in pair[k]]
                options = 1
                for i in range(N_Loc):
                    options *= len(splits[i])
                if options < cutoff:
                    # Cartesian product, first locus slowest (cutils.open_ambiguities order)
                    sides.append([[list(c) for c in itertools.product(*splits[:N_Loc])]])
                else:
                    sides.append([])
            if sides[0] and sides[1]:
                phases.append([sides[0], sides[1]])
        return phases

    # ------------------------------------------------------------------ native text pipeline
    def _text_handle(self):
        """GrimbText: dictionaries + priority parameters for the C++ tokeniser / formatter."""
        if getattr(self, "_text", None) is not None:
            return self._text
        g = self.netGraph
        lib = g.lib
        d = _lib.TextDesc()
        d.n_loci, d.n_pops = self.L, self.P
        keep = []

        def cstrings(items):
            arr = (C.c_char_p * max(1, len(items)))(*[s.encode("utf8") for s in items])
            keep.append(arr)
            return arr

        d.locus_names = cstrings(self.loci)
        d.allele_names = cstrings([a for l in range(self.L) for a in g.alleles[l]])
        counts = (C.c_int32 * self.L)(*[len(g.alleles[l]) for l in range(self.L)])
        cbp = (C.c_double * self.P)(*[float(x) for x in self.count_by_prob])
        keep.extend([counts, cbp])
        d.allele_counts, d.pop_names, d.count_by_prob = counts, cstrings(self.populations), cbp
        pr = self.priority
        d.alpha, d.eta, d.beta, d.gamma, d.delta = (float(pr[k]) for k in ("alpha", "eta", "beta", "gamma", "delta"))
        d.unk_priors_mr = 1 if self.unk_priors == "MR" else 0
        for l in range(self.L):
            d.key_bits[l] = g.key_bits[l]
        d.n_threads = int(os.environ.get("GRIMB_HOST_THREADS", "0"))
        if self.type_allowed is not None:
            keep.append(self.type_allowed)
            d.type_allowed = self.type_allowed.ctypes.data
        h = C.c_void_p()
        _lib.check(lib.grimb_text_create(C.byref(d), C.byref(h)), "grimb_text_create", lib)
        self._text = h
        return h

    @staticmethod
    def _byte_chunks(f, max_bytes=None):
        """Yields (bytes of whole lines, number of lines before them) from a binary file, reading big
        blocks and cutting at the last newline -- no per-line work in Python."""
        max_bytes = max_bytes or int(os.environ.get("GRIMB_TEXT_BYTES", str(24 << 20)))
        first = 0
        carry = b""
        while True:
            block = f.read(max_bytes)
            if not block:
                break
            data = carry + block if carry else block
            cut = data.rfind(b"\n")
            if cut < 0:
                carry = data
                continue
            chunk, carry = data[:cut + 1], data[cut + 1:]
            yield chunk, first
            first += chunk.count(b"\n")
        if carry:
            yield carry, first

    def impute_text_stream(self, data, first_index=0, max_bytes=None):
        """impute_text over a large bytes object in bounded pieces; returns the six texts."""
        import io
        parts = {k: [] for k in _lib.OUT_KEYS}
        for chunk, first in self._byte_chunks(io.BytesIO(data), max_bytes):
            out = self.impute_text(chunk, first_index + first)
            for k in _lib.OUT_KEYS:
                parts[k].append(out[k])
        return {k: b"".join(v) for k, v in parts.items()}

    def impute_text(self, data, first_index=0):
        """bytes of input lines -> dict of the six output texts (bytes), through grimb_impute_text."""
        lib = self.netGraph.lib
        t = self._text_handle()
        engines = (C.c_void_p * len(self.workspaces))(*[self.netGraph.engine(w) for w in self.workspaces[:1]])
        # engines of the bigger tiers are created lazily: pass only what exists, retry on overflow
        n_eng = 1
        out = _lib.TextOut()
        while True:
            rc = lib.grimb_impute_text(t, engines, n_eng, C.byref(self.cfg), data, len(data), first_index, C.byref(out))
            if rc == -3 and n_eng < len(self.workspaces):   # GRIMB_E_NOMEM: a subject overflowed the last tier
                engines[n_eng] = self.netGraph.engine(self.workspaces[n_eng])
                n_eng += 1
                continue
            _lib.check(rc, "grimb_impute_text", lib)
            break
        self.stats["subjects"] += out.n_lines
        self.stats["pair_evals"] += out.pair_evals
        self.stats["workspace_retries"] += out.workspace_retries
        for k in range(4):
            self.stats["plan"][k] += out.plan_count[k]
        for k, v in (("tokenise_seconds", out.seconds_tokenise), ("abi_seconds", out.seconds_gpu),
                     ("format_seconds", out.seconds_format)):
            self.stats[k] = self.stats.get(k, 0.0) + v
        return {k: C.string_at(out.data[i], out.size[i]) for i, k in enumerate(_lib.OUT_KEYS)}

    def impute_file_sharded(self, in_path, out_paths, chunk_bytes, rank, world, board_path, n_tiers=1):
        """This rank's share of one input file (chunks rank, rank + world, ...), streamed into the shared final files
        at the offsets the ranks agree on through the board file (include/grimb200.h: grimb_impute_file_sharded).
        n_tiers: workspace tiers to offer (a subject that overflows the last one fails the call with
        GRIMB_E_NOMEM; the caller restarts all ranks with one more tier)."""
        lib = self.netGraph.lib
        t = self._text_handle()
        n_eng = max(1, min(n_tiers, len(self.workspaces)))
        engines = (C.c_void_p * len(self.workspaces))(*[self.netGraph.engine(w) for w in self.workspaces[:n_eng]])
        paths = (C.c_char_p * 6)(*[(out_paths[k].encode("utf8") if k in out_paths else None) for k in _lib.OUT_KEYS])
        st = _lib.FileStats()
        self.cfg.hap_pop_pair = 0
        self.cfg.em = 0
        rc = lib.grimb_impute_file_sharded(t, engines, n_eng, C.byref(self.cfg), in_path.encode("utf8"), paths, chunk_bytes,
                                           rank, world, board_path.encode("utf8"), C.byref(st))
        _lib.check(rc, "grimb_impute_file_sharded", lib)
        self.stats["subjects"] += st.n_lines
        self.stats["pair_evals"] += st.pair_evals
        self.stats["workspace_retries"] += st.workspace_retries
        for k in range(4):
            self.stats["plan"][k] += st.plan_count[k]
        return st

    def impute_file_native(self, in_path, out_paths=None, byte_lo=0, byte_hi=-1, first_index=0, chunk_bytes=0):
        """The whole file (or the lines starting in [byte_lo, byte_hi)) through grimb_impute_file: memory-mapped
        input, tokenise | GPU | format | write overlapped on host threads.  out_paths: dict key -> path of the
        outputs to stream to files; the others are returned as bytes.  -> (dict of bytes, _lib.FileStats)."""
        lib = self.netGraph.lib
        t = self._text_handle()
        chunk_bytes = chunk_bytes or int(os.environ.get("GRIMB_FILE_CHUNK", "0"))
        engines = (C.c_void_p * len(self.workspaces))(*[self.netGraph.engine(w) for w in self.workspaces[:1]])
        n_eng = 1
        paths = (C.c_char_p * 6)(*[(out_paths[k].encode("utf8") if out_paths and out_paths.get(k) else None)
                                   for k in _lib.OUT_KEYS])
        out, st = _lib.TextOut(), _lib.FileStats()
        while True:
            rc = lib.grimb_impute_file(t, engines, n_eng, C.byref(self.cfg), in_path.encode("utf8"), byte_lo, byte_hi,
                                       first_index, paths, chunk_bytes, C.byref(out), C.byref(st))
            if rc == -3 and n_eng < len(self.workspaces):   # GRIMB_E_NOMEM: a subject overflowed the last tier
                engines[n_eng] = self.netGraph.engine(self.workspaces[n_eng])
                n_eng += 1
                continue
            _lib.check(rc, "grimb_impute_file", lib)
            break
        self.stats["subjects"] += st.n_lines
        self.stats["pair_evals"] += st.pair_evals
        self.stats["workspace_retries"] += st.workspace_retries
        for k in range(4):
            self.stats["plan"][k] += st.plan_count[k]
        for k, v in (("tokenise_seconds", st.seconds_tokenise), ("abi_seconds", st.seconds_gpu),
                     ("format_seconds", st.seconds_format), ("write_seconds", st.seconds_write)):
            self.stats[k] = self.stats.get(k, 0.0) + v
        self._last_file_out = out   # keeps the pointers' owner (the GrimbText) in view; valid until the next call
        return out, st

    def impute_file(self, config, planb=None, em_mr=False, em=False):
        """Reads config["imputation_input_file"], writes the six output files
        (impute.py:1985-2155 of the reference)."""
        # the planb argument overrides the configuration for this call only (impute.py:1985,2046 of the reference)
        eff_planb = bool(config["planb"]) if planb is None else bool(planb)
        saved = (self.cfg.planb, self.config["planb"])
        self.cfg.planb = 1 if eff_planb else 0
        if self.config["planb"] != eff_planb:
            self.config = dict(self.config, planb=eff_planb)   # the numpy front end classifies foreign loci by it
        try:
            self._impute_file(config, em_mr, em)
        finally:
            self.cfg.planb = saved[0]
            if self.config["planb"] != saved[1]:
                self.config = dict(self.config, planb=saved[1])

    def _impute_file(self, config, em_mr, em):
        targets = {"miss": "imputation_out_miss_file", "problem": "imputation_out_problem_file"}
        # the EM-facing modes (hap_pop_pair rows, em, per-subject phase masks) go through the numpy
        # host front end; the C++ text pipeline serves the default mode
        special = bool(em_mr or em or self.phase_masks is not None)
        self._em_mr = False
        self.cfg.hap_pop_pair = 0
        self.cfg.em = 0
        if os.environ.get("GRIMB_PY_HOST") != "1" and not special:
            # native host pipeline: C++ tokeniser / formatter around the kernels (grimb_impute_text)
            if config["output_MUUG"]:
                targets["umug"] = "imputation_out_umug_freq_file"
                targets["umug_pops"] = "imputation_out_umug_pops_file"
            if config["output_haplotypes"]:
                targets["pmug"] = "imputation_out_hap_freq_file"
                targets["pmug_pops"] = "imputation_out_hap_pops_file"
            # outputs that are switched off are produced empty by the formatter and discarded
            self.impute_file_native(config["imputation_input_file"], {k: config[ck] for k, ck in targets.items()})
            return
        with open(config["imputation_input_file"]) as f:
            files = self.impute_lines(f, em_mr=em_mr, em=em)
        if config["output_MUUG"]:
            targets["umug"] = "imputation_out_umug_freq_file"
            targets["umug_pops"] = "imputation_out_umug_pops_file"
        if config["output_haplotypes"]:
            targets["pmug"] = "imputation_out_hap_freq_file"
            targets["pmug_pops"] = "imputation_out_hap_pops_file"
        for k, ck in targets.items():
            with open(config[ck], "w") as f:
                f.writelines(files[k])


def _phase_mask(bits):
    """A bin_imputation_in_file entry (one 0/1 per typed locus) -> the GrimbBatch.phase_mask word."""
    pm = 0
    for m, e in enumerate(bits):
        if e == 1 and m < 16:
            pm |= 1 << m
    return pm


_SUBJECT_FIELDS = ("status", "plan_umug", "plan_pmug", "flags", "tot_umug", "tot_pmug")


def _splice_rows(base, part, idx):
    """Rows of the whole batch with the subjects `idx` (CUDA int64) taken from `part` (their re-issue)."""
    import torch
    out = {"pair_evals": base["pair_evals"] + part["pair_evals"]}
    for f in _SUBJECT_FIELDS:
        out[f] = base[f].clone()
        out[f][idx] = part[f]
    S, dev = base["status"].shape[0], base["status"].device
    pos = torch.full((S,), -1, dtype=torch.int64, device=dev)
    pos[idx] = torch.arange(idx.numel(), device=dev)
    for k in _lib.ROW_KINDS:
        bo, po = base[k + "_off"], part[k + "_off"]
        cnt = bo[1:] - bo[:-1]
        cnt[idx] = po[1:] - po[:-1]
        off = torch.zeros(S + 1, dtype=torch.int64, device=dev)
        torch.cumsum(cnt, 0, out=off[1:])
        total = int(off[-1])
        owner = torch.repeat_interleave(torch.arange(S, device=dev), cnt, output_size=total)
        within = torch.arange(total, device=dev) - off[owner]
        p = pos[owner]
        mine = p >= 0
        rows = torch.empty((total,) + tuple(base[k].shape[1:]), dtype=base[k].dtype, device=dev)
        prob = torch.empty(total, dtype=torch.float64, device=dev)
        src = po[p[mine]] + within[mine]
        rows[mine], prob[mine] = part[k][src], part[k + "_prob"][src]
        psrc = src
        src = bo[owner[~mine]] + within[~mine]
        rows[~mine], prob[~mine] = base[k][src], base[k + "_prob"][src]
        out[k], out[k + "_prob"], out[k + "_off"] = rows, prob, off
        if k == "pmug" and "pmug_pairs" in base:
            pairs = torch.empty((total, 2), dtype=base["pmug_pairs"].dtype, device=dev)
            pairs[mine], pairs[~mine] = part["pmug_pairs"][psrc], base["pmug_pairs"][src]
            out["pmug_pairs"] = pairs
    return out


class GenotypeResults(object):
    """Result of Imputation.impute_genotypes / impute_genotype_lists: ragged rows in input order (include/grimb200.h,
    GrimbRows).

    Per subject [S]: status (GRIMB_ST_*), plan_umug, plan_pmug (GRIMB_PLAN_*), tot_umug, tot_pmug (the counts the
    reference prints), flags (bit 0 has results, bit 1 written to .miss, bit 2 written to .problem).
    Per row kind k in ("umug", "pmug", "umug_pops", "pmug_pops"): k_off [S+1] (int64; subject s owns rows
    k_off[s]:k_off[s+1], in rank order), k (uint16 rows: umug [n][L][2] (min id, max id) allele pairs, pmug [n][2][L]
    haplotype 1 / haplotype 2 (0 = no allele), pop kinds [n][2] population indices, 0xFFFF = all_pops) and k_prob
    [n] (float64).  alleles[l][id - 1] names table allele `id` of locus l; populations[p] names population p.
    pmug_pairs [n_pmug][2]: under em_mr (impute_genotype_lists), the populations of haplotype 1 and haplotype 2 of
    each PMUG row (the hap;pop pairs of the reference's hap_pop_pair output); None otherwise.
    pair_evals: pair evaluations of the batch; workspace_retries: subjects re-issued on a bigger workspace tier;
    capacity_reruns: times the imputation ran again because its result arrays were too small (0 normally).
    Arrays are CUDA tensors when the input was one, numpy arrays otherwise."""

    def __init__(self, d, alleles, populations, workspace_retries, as_numpy):
        import torch
        self.alleles, self.populations = alleles, populations
        self.pair_evals, self.workspace_retries = d["pair_evals"], workspace_retries
        self.capacity_reruns = d["capacity_reruns"]
        for f in _SUBJECT_FIELDS:
            v = d[f]   # uint8, or int32 storage of the uint32 totals
            if as_numpy:
                v = v.cpu().numpy()
                setattr(self, f, v.view(np.uint32) if v.dtype == np.int32 else v)
            else:
                setattr(self, f, v.view(torch.uint32) if v.dtype == torch.int32 else v)
        for k in _lib.ROW_KINDS:
            rows = d[k]
            setattr(self, k, rows.cpu().numpy().view(np.uint16) if as_numpy else rows.view(torch.uint16))
            setattr(self, k + "_prob", d[k + "_prob"].cpu().numpy() if as_numpy else d[k + "_prob"])
            setattr(self, k + "_off", d[k + "_off"].cpu().numpy() if as_numpy else d[k + "_off"])
        pp = d.get("pmug_pairs")
        self.pmug_pairs = None if pp is None else (pp.cpu().numpy().view(np.uint16) if as_numpy else pp.view(torch.uint16))

    def __len__(self):
        return int(self.status.shape[0])
