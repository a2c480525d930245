#!/usr/bin/env python
"""bench.py -- BASELINE.json metric: subjects/sec (+ hap-pair evals/sec) of the per-subject
imputation hot path on N B200s, beside the CPU port of the reference on the host cores.

Workload (BASELINE.json configs[1], SURVEY 8(d) "C2"): S = 2^20 synthetic, fully typed,
unambiguous 5-locus subjects, one population, haplotypes drawn proportional to frequency from
a synthetic Zipf table of N_full = 1M haplotypes (alleles/locus 700/1200/600/250/700, seed
20261018; subjects seed 1), minimal-configuration keys with number_of_results 10, UMUG + PMUG
outputs, Plan B on.  One step = one pass of the hot path over the whole batch.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--subjects S] [--haps H]
                  [--dump-outputs DIR]

value  : subjects/s, batch already resident in HBM, CUDA-event timed (max over ranks)
e2e    : same through grimb_impute_host with pinned HOST buffers (H2D + kernel + D2H per step)
roofline / cpu_baseline: see DESIGN.md "Measurement".  roofline.probe_bound places the dominant kernel against
the random 32-byte-sector rate measured by tools/sector_peak.cu (the probe-bound roofline); e2e.link places the
host-buffer leg against the time the PCIe link alone needs for the same bytes (tools/pcie_peak.py).
--dump-outputs DIR: the results of the last timed `value` step (rank 0's batch) as DIR/*.npy, see dump_outputs().
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (os.path.join(ROOT, "py-graph-imputation_b200"), os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

LOCI = ["A", "B", "C", "DQB1", "DRB1"]
N_ALLELES = [700, 1200, 600, 250, 700]
TABLE_SEED = 20261018
SUBJECT_SEED = 1


# --------------------------------------------------------------------------- workload
def make_table(n_full):
    """-> (allele names per locus, full_alleles uint16 [N][5] (1-based ids), freqs [N][1])."""
    rng = np.random.RandomState(TABLE_SEED)
    cols = []
    for na in N_ALLELES:
        w = 1.0 / np.arange(1, na + 1) ** 1.1
        w /= w.sum()
        cols.append(rng.choice(na, size=int(n_full * 1.25) + 1000, p=w))
    tup = np.stack(cols, axis=1).astype(np.int64)
    packed = np.zeros(len(tup), np.int64)
    for l in range(5):
        packed = packed * 2048 + tup[:, l]
    _u, first = np.unique(packed, return_index=True)
    tup = tup[np.sort(first)][:n_full]
    n = len(tup)
    f = 1.0 / np.arange(1, n + 1)
    f /= f.sum()
    names = [["%s*%02d:%02d" % (loc, a // 60 + 1, a % 60 + 1) for a in range(na)] for loc, na in zip(LOCI, N_ALLELES)]
    return names, (tup + 1).astype(np.uint16), f.reshape(n, 1).astype(np.float64)


def pack_batch(alleles, key_bits, n_alleles):
    """ABI v4 packed form of fully typed, unambiguous subjects: [S][2] keys (side-0 / side-1 alleles packed with
    the tables' key layout) + [S] flag words (bits 0-4 heterozygous, 5-9 / 10-14 allele absent from the table)."""
    S, L = alleles.shape[0], alleles.shape[1]
    keys = np.zeros((S, 2), np.uint64)
    flags = np.zeros(S, np.uint16)
    shift = 0
    for l in range(L):
        a0, a1 = alleles[:, l, 0].astype(np.uint64), alleles[:, l, 1].astype(np.uint64)
        keys[:, 0] |= a0 << np.uint64(shift)
        keys[:, 1] |= a1 << np.uint64(shift)
        flags |= ((a0 != a1).astype(np.uint16) << l) | ((a0 > n_alleles[l]).astype(np.uint16) << (5 + l)) \
            | ((a1 > n_alleles[l]).astype(np.uint16) << (10 + l))
        shift += int(key_bits[l])
    return np.ascontiguousarray(keys.reshape(-1)), flags


def make_subjects(full_alleles, freqs, n_subj, seed):
    """Encoded batch (GrimbBatch arrays) of fully typed unambiguous subjects."""
    rng = np.random.RandomState(seed)
    p = freqs[:, 0] / freqs[:, 0].sum()
    idx = rng.choice(len(p), size=(n_subj, 2), p=p)
    flip = rng.rand(n_subj, 5) < 0.5
    h1 = full_alleles[idx[:, 0]]
    h2 = full_alleles[idx[:, 1]]
    a = np.where(flip, h2, h1)
    b = np.where(flip, h1, h2)
    alleles = np.stack([a, b], axis=2).astype(np.uint16)          # [S][L][2]
    # ABI v4: one allele per typed side everywhere -> no `counts`; one prior matrix -> no `prior_index`
    batch = {
        "typed_mask": np.full(n_subj, 31, np.uint16),
        "allele_off": (np.arange(n_subj + 1, dtype=np.uint64) * 10).astype(np.uint32),
        "alleles": np.ascontiguousarray(alleles.reshape(-1)),
        "priors": np.ones((1, 1, 1), np.float64),
    }
    return batch, alleles


def subject_lines(names, alleles, lo, hi):
    out = []
    for s in range(lo, hi):
        gl = "^".join(names[l][alleles[s, l, 0] - 1] + "+" + names[l][alleles[s, l, 1] - 1] for l in range(5))
        out.append("S%d,%s,CAU,CAU\n" % (s, gl))
    return out


def base_conf():
    conf = json.load(open(os.path.join(ROOT, "tests", "golden", "data", "base_conf.json")))
    conf["number_of_results"] = 10
    return conf


# --------------------------------------------------------------------------- CPU port (oracle)
class _FullOnlyGraph(object):
    """Oracle-side store holding only what fully typed subjects probe (the full-label dict).
    The reference's Graph would hold every marginal too (~30x more nodes); for this workload
    Plan A always hits, so per-subject CPU work is identical and the (untimed) build stays
    feasible in pure Python."""

    def __init__(self, names, full_alleles, freqs):
        import grim_oracle as go
        self.full_label = "12345"
        self.pops = ["CAU"]
        self.node = {}
        self.names = []
        cols = [np.array(names[l], dtype=object)[full_alleles[:, l] - 1] for l in range(5)]
        for i in range(len(full_alleles)):
            nm = "~".join(c[i] for c in cols)
            self.node[nm] = ("12345", [float(freqs[i, 0])], i)
        self.adjs_query = go.OracleGraph.adjs_query.__get__(self)
        self.node_probs = go.OracleGraph.node_probs.__get__(self)
        self.toplinks = {}
        self.conn = {}
        self.by_label = {}


def cpu_port_rate(g, lines, procs):
    """subjects/s of the oracle port on `procs` forked processes over `lines`."""
    import multiprocessing as mp

    import grim_oracle as go
    cfg = go.load_config(base_conf())
    n_sample = len(lines)
    chunks = [lines[i::procs] for i in range(procs)]

    def work(ch, q):
        imp = go.OracleImputation(g, cfg, np.ones(1))
        t = time.time()
        out = imp.impute_lines(ch)
        q.put((time.time() - t, imp.pair_evals, out["umug"].count("\n"), out["problem"].count("\n")))

    q = mp.Queue()
    t0 = time.time()
    ps = [mp.Process(target=work, args=(ch, q)) for ch in chunks]
    for p_ in ps:
        p_.start()
    res = [q.get() for _ in ps]
    for p_ in ps:
        p_.join()
    wall = time.time() - t0
    evals = sum(r[1] for r in res)
    return n_sample / wall, evals / wall, wall, sum(r[3] for r in res)


# --------------------------------------------------------------------------- clocks
class ClockSampler(threading.Thread):
    def __init__(self, gpu):
        super().__init__(daemon=True)
        self.gpu = gpu
        self.rows = []
        self.stop_flag = False

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self.stop_flag:
            try:
                o = subprocess.run(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                   capture_output=True, text=True, timeout=5).stdout.strip()
                if o:
                    self.rows.append([x.strip() for x in o.split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        sm = sorted(int(r[0]) for r in self.rows if r[0].isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i].startswith("Active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None,
                "sm_max_mhz": int(self.rows[0][1]) if self.rows[0][1].isdigit() else None, "reasons": reasons}


# --------------------------------------------------------------------------- reference arm
def _reference_graph(names, full_alleles, freqs):
    """The UNMODIFIED reference's Graph (oracle/_ref/grim/imputation/networkx_graph.py), filled in memory with
    the full-haplotype nodes of the synthetic table instead of being loaded from nodes/edges CSV files (the
    reference's own generator needs ~10 minutes for a table of this size).  Every subject of this workload is
    served by Plan A, whose only store access is the full-label dict lookup of Graph.adjs_query, so the
    per-subject work the reference performs is unchanged."""
    from grim.imputation.networkx_graph import Graph
    g = Graph({"full_loci": "12345", "nodes_for_plan_A": []})
    cols = [np.array(names[l], dtype=object)[full_alleles[:, l] - 1] for l in range(5)]
    verts = []
    for i in range(len(full_alleles)):
        nm = "~".join(c[i] for c in cols)
        g.Vertices_attributes[nm] = ("12345", [float(freqs[i, 0])], i)
        verts.append(nm)
    g.Whole_Vertices_attributes = g.Vertices_attributes
    g.Vertices = np.array(verts, dtype=np.object_)
    g.Whole_Vertices = g.Vertices
    g.Edges = np.zeros(0, np.uint32)
    g.Whole_Edges = np.zeros(0, np.uint32)
    g.Neighbors_start = np.zeros(len(verts) + 1, np.uint32)
    g.Whole_Neighbors_start = g.Neighbors_start
    return g


def reference_rate(g, lines, procs):
    """subjects/s of the reference's own Imputation.impute_file over `lines`, one forked process per core on
    a contiguous chunk with the graph inherited by fork (the strategy of the reference's scripts/runfile_mp.py)."""
    import contextlib
    import multiprocessing as mp
    import tempfile

    from grim.imputation.impute import Imputation
    tmp = tempfile.mkdtemp(prefix="grimref_")
    conf = base_conf()
    per = (len(lines) + procs - 1) // procs

    def work(w, q):
        sub = lines[w * per:(w + 1) * per]
        inp = os.path.join(tmp, "in%d.csv" % w)
        with open(inp, "w") as f:
            f.writelines(sub)
        lm = dict(conf["loci_map"])
        config = {
            "planb": True, "pops": conf["populations"], "priority": conf["priority"], "epsilon": conf["epsilon"],
            "number_of_results": conf["number_of_results"], "number_of_pop_results": conf["number_of_pop_results"],
            "output_MUUG": True, "output_haplotypes": True, "imputation_input_file": inp,
            "imputation_out_umug_freq_file": os.path.join(tmp, "o%d.umug" % w),
            "imputation_out_umug_pops_file": os.path.join(tmp, "o%d.umug.pops" % w),
            "imputation_out_hap_freq_file": os.path.join(tmp, "o%d.pmug" % w),
            "imputation_out_hap_pops_file": os.path.join(tmp, "o%d.pmug.pops" % w),
            "imputation_out_miss_file": os.path.join(tmp, "o%d.miss" % w),
            "imputation_out_problem_file": os.path.join(tmp, "o%d.problem" % w),
            "factor_missing_data": conf.get("factor_missing_data", 0.01), "loci_map": lm,
            "matrix_planb": conf["Plan_B_Matrix"], "pops_count_file": "", "use_pops_count_file": False,
            "number_of_options_threshold": 100000, "max_haplotypes_number_in_phase": 100,
            "bin_imputation_input_file": "None", "nodes_for_plan_A": [], "save_mode": False, "UNK_priors": "MR",
            "full_loci": "12345",
        }
        imp = Imputation(g, config)
        t = time.time()
        with open(os.devnull, "w") as null, contextlib.redirect_stdout(null):   # two prints + a timing per subject
            imp.impute_file(config)
        rows = sum(1 for _ in open(config["imputation_out_umug_freq_file"]))
        prob = sum(1 for _ in open(config["imputation_out_problem_file"]))
        q.put((time.time() - t, rows, prob))

    q = mp.Queue()
    t0 = time.time()
    ps = [mp.Process(target=work, args=(w, q)) for w in range(procs) if w * per < len(lines)]
    for p_ in ps:
        p_.start()
    res = [q.get() for _ in ps]
    for p_ in ps:
        p_.join()
    wall = time.time() - t0
    import shutil
    shutil.rmtree(tmp, ignore_errors=True)
    if sum(r[1] for r in res) < len(lines) * 0.9 or sum(r[2] for r in res):
        raise RuntimeError("the reference did not impute the sample: %s" % (res[:3],))
    return len(lines) / wall, wall


def run_reference(args, rank):
    if rank != 0:
        return
    names, fa, ff = make_table(args.haps)
    _batch, alleles = make_subjects(fa, ff, args.subjects, SUBJECT_SEED)
    cores = os.cpu_count() or 1
    n_sample = min(args.subjects, args.ref_sample * cores)
    lines = subject_lines(names, alleles, 0, n_sample)
    ref_dir = os.path.join(ROOT, "oracle", "_ref")
    kind = "port"
    if os.path.isdir(os.path.join(ref_dir, "grim")):
        # the reference itself, vendored by oracle/build_ref.sh (no product module is imported in this arm)
        sys.path.insert(0, ref_dir)
        try:
            g = _reference_graph(names, fa, ff)
            reference_rate(g, lines[:cores * 8], cores)     # import / fork check
            kind = "reference"
        except Exception as exc:   # e.g. a Python minor version the prebuilt cutils does not load on
            sys.stderr.write("reference arm: falling back to the port (%r)\n" % (exc,))
            sys.path.remove(ref_dir)
    if kind == "port":
        g = _FullOnlyGraph(names, fa, ff)
    vals = []
    for _ in range(args.warmup + args.steps):
        if kind == "reference":
            rate, wall = reference_rate(g, lines, cores)
            erate = 0.0
        else:
            rate, erate, wall, prob = cpu_port_rate(g, lines, cores)
        vals.append((rate, erate, wall))
    vals = vals[args.warmup:]
    rate = float(np.mean([v[0] for v in vals]))
    line = {
        "impl": "reference", "metric": "subjects_per_sec", "value": rate, "unit": "subjects/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 * float(np.mean([v[2] for v in vals])),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "pair_evals_per_sec": (float(np.mean([v[1] for v in vals])) if kind == "port" else None),
        "config": workload_config(args),
        "cpu_baseline": {"value": rate, "unit": "subjects/s", "cores": cores, "kind": kind,
                         "sample": ("first %d of the %d subjects, %d forked processes, " % (n_sample, args.subjects, cores))
                         + ("the unmodified reference (oracle/_ref, vendored by oracle/build_ref.sh): its own "
                            "Imputation.impute_file per chunk, Graph filled in memory with the table's full-haplotype nodes"
                            if kind == "reference" else "oracle/grim_oracle.py (oracle/_ref absent)")},
        "e2e": {"value": rate, "unit": "subjects/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


DUMP_MAX_SUBJECTS = 1 << 17     # ~29 MB of .npy files
DUMP_SEED = 20261020


def dump_outputs(out_dir, comp, words, pair_evals):
    """Writes what one grimb_impute_device call returned for the batch, decoded per subject, so that two builds
    can be compared file for file: word offsets come from an atomic cursor and differ from run to run, so the
    files hold each subject's values, not the raw arrays.  Subjects: all of them, or a fixed seeded sample of
    DUMP_MAX_SUBJECTS for larger batches (subject_index.npy).  Every subject of this workload is fully typed
    with one population, i.e. a SIMPLE record (include/grimb200.h); any other kind is an error.
      status [n], has_results [n], umug_prob [n] (the UMUG genotype's probability), pmug_rows [n],
      pmug_phase [n][16] (phase id of PMUG row k in rank order, -1 past pmug_rows), pmug_prob [n][16] (0 past
      pmug_rows), pair_evals [1]."""
    from grim.imputation import _lib
    S = len(comp)
    idx = np.arange(S) if S <= DUMP_MAX_SUBJECTS else \
        np.sort(np.random.RandomState(DUMP_SEED).choice(S, DUMP_MAX_SUBJECTS, replace=False))
    c = comp[idx]
    n = len(idx)
    wf = words.view(np.float64)
    rows = np.zeros(n, np.float32)
    phase = np.full((n, 16), -1.0, np.float32)
    prob = np.zeros((n, 16), np.float64)
    for i in range(n):
        kf, off = int(c["kind_flags"][i]), int(c["off"][i])
        if (kf & 3) != _lib.KIND_SIMPLE:
            raise RuntimeError("--dump-outputs: subject %d is not a SIMPLE record (kind_flags %#x)" % (idx[i], kf))
        k = kf >> 4
        if k == 15:        # long form: a count word, a word of phase ids, then the probabilities
            k = min(16, int(words[off]))
            ph, pr = int(words[off + 1]), wf[off + 2:off + 2 + k]
        else:
            ph, pr = int(c["phases"][i]), (wf[off:off + k] if kf & _lib.KIND_WORDS else c["total"][i])
        rows[i] = k
        phase[i, :k] = [(ph >> (4 * q)) & 15 for q in range(k)]
        prob[i, :k] = pr
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"subject_index": idx.astype(np.float64), "status": c["status"].astype(np.float32),
              "has_results": ((c["kind_flags"] & _lib.KIND_HAS_RESULTS) != 0).astype(np.float32),
              "umug_prob": c["total"].astype(np.float64), "pmug_rows": rows, "pmug_phase": phase, "pmug_prob": prob,
              "pair_evals": np.array([pair_evals], np.float64)}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def workload_config(args):
    return {"workload": "C2: %d fully typed unambiguous 5-locus subjects, 1 population, synthetic Zipf table of %d "
                        "haplotypes, UMUG+PMUG top-10, Plan B on" % (args.subjects, args.haps),
            "subjects_per_gpu": args.subjects, "table_haplotypes": args.haps,
            "l2": "inputs + tables exceed L2 (no flush needed)"}


# --------------------------------------------------------------------------- GPU arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--subjects", type=int, default=1 << 20)
    ap.add_argument("--haps", type=int, default=1000000)
    ap.add_argument("--ref-sample", type=int, default=2500, help="CPU port: subjects per core per step")
    ap.add_argument("--cpu-sample", type=int, default=12000, help="cpu_baseline: subjects on 1 core")
    ap.add_argument("--text-subjects", type=int, default=1 << 18, help="subjects of the text-to-text measurement")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the C3 / C4 / C5 / K0 sub-records")
    ap.add_argument("--c3-subjects", type=int, default=1 << 18)
    ap.add_argument("--c4-subjects", type=int, default=4000)
    ap.add_argument("--c4-heavy-subjects", type=int, default=400)
    ap.add_argument("--c4-wide-subjects", type=int, default=16)
    ap.add_argument("--c5-haps", type=int, default=100000)
    ap.add_argument("--c5-subjects", type=int, default=1 << 16)
    ap.add_argument("--c5m-haps", type=int, default=2000000, help="nine-locus table under a Plan_A_Matrix (0: skip)")
    ap.add_argument("--config-sample", type=int, default=300, help="subjects per configuration checked against the oracle")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the results of the last timed step as DIR/*.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the GPU path")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return

    import torch
    import torch.distributed as dist
    from grim.imputation import _lib
    from grim.imputation.impute import make_config
    from grim.imputation.networkx_graph import Graph
    from grim.run_impute_def import load_config

    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa_cpus = None
    if world > 1 and os.environ.get("GRIMB_NUMA_BIND", "1") != "0":
        from grim.imputation.multi_gpu import bind_to_device_numa_node
        numa_cpus = bind_to_device_numa_node(local)   # before any pinned allocation
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.load()
    conf = load_config(base_conf())
    names, fa, ff = make_table(args.haps)

    # ---- tables: built once on rank 0, replicated with one NCCL broadcast of the device image
    g = Graph(conf, device=local)
    t_build = time.time()
    if rank == 0:
        g.from_arrays(names, fa, ff)
    if world > 1:
        size = torch.zeros(1, dtype=torch.int64, device=dev)
        if rank == 0:
            nbytes = C.c_int64()
            _lib.check(lib.grimb_tables_image_size(g.handle, C.byref(nbytes)), "image_size")
            size[0] = nbytes.value
        dist.broadcast(size, 0)
        nb = int(size.item())
        if rank == 0:
            ptr = C.c_void_p()
            _lib.check(lib.grimb_tables_image_ptr(g.handle, C.byref(ptr)), "image_ptr")

            class _View(object):
                __cuda_array_interface__ = {"shape": (nb,), "typestr": "|u1", "data": (ptr.value, False), "version": 2}
            img = torch.as_tensor(_View(), device=dev)
        else:
            img = torch.empty(nb, dtype=torch.uint8, device=dev)
        dist.broadcast(img, 0)
        torch.cuda.synchronize()
        if rank != 0:
            g._set_dictionaries(names)
            h = C.c_void_p()
            _lib.check(lib.grimb_tables_from_image(C.c_void_p(img.data_ptr()), nb, local, C.byref(h)), "from_image")
            g.handle = h
            del img
    t_build = time.time() - t_build
    info = g.info()

    # ---- subjects: every rank imputes its own shard (weak scaling: S per GPU)
    batch, alleles = make_subjects(fa, ff, args.subjects, SUBJECT_SEED + rank)
    S = args.subjects
    cfg = make_config(conf, LOCI, 1)
    eng = g.engine(8 << 20)

    def tens(a, pin=False):
        t = torch.from_numpy(a)
        return t.pin_memory() if pin else t

    # the batch in the packed form of ABI v4 (18 bytes per subject: two packed keys + a flag word), which is
    # what the tokeniser emits for input of this shape; GRIMB_BENCH_PACKED=0 measures the general form
    use_packed = os.environ.get("GRIMB_BENCH_PACKED", "1") != "0"
    if use_packed:
        pk, pf = pack_batch(alleles, g.key_bits, [len(a) for a in names])
        batch = {"packed_keys": pk.view(np.int64), "packed_flags": pf, "priors": batch["priors"]}
        keys_in = ["packed_keys", "packed_flags", "priors"]
    else:
        keys_in = ["typed_mask", "allele_off", "alleles", "priors"]
    # result capacities: 16-byte records for everybody, a few 8-byte words for subjects with several accepted
    # phases, and room for the subjects the general kernel serves (none in this workload)
    word_cap, gen_cap, hap_cap, pop_cap = S * 2, S // 8 + 1024, S // 4 + 1024, S // 4 + 1024
    SZ = {"compact": 16, "words": 8, "general": 48, "hap_rows": 24, "pop_rows": 16}
    CAP = {"compact": S, "words": word_cap, "general": gen_cap, "hap_rows": hap_cap, "pop_rows": pop_cap}

    def make_structs(inputs, outs, totals):
        b = _lib.Batch()
        b.n_subjects = S
        for k in keys_in:
            setattr(b, k, inputs[k].data_ptr())
        b.n_alleles_total = 0 if use_packed else S * 10
        b.n_priors = 1
        r = _lib.Results()
        r.compact = outs["compact"].data_ptr()
        r.words, r.word_capacity = outs["words"].data_ptr(), word_cap
        r.general, r.general_capacity = outs["general"].data_ptr(), gen_cap
        r.hap_rows, r.hap_capacity = outs["hap_rows"].data_ptr(), hap_cap
        r.pop_rows, r.pop_capacity = outs["pop_rows"].data_ptr(), pop_cap
        r.totals = totals.ctypes.data
        return b, r

    def as_signed(a):
        return a.view(np.int16) if a.dtype == np.uint16 else a.view(np.int32) if a.dtype == np.uint32 else a

    # device-resident leg
    d_in = {k: tens(as_signed(batch[k])).to(dev) for k in keys_in}
    d_out = {k: torch.zeros(CAP[k] * SZ[k], dtype=torch.uint8, device=dev) for k in SZ}
    tot_dev = np.zeros(9, np.int64)
    db, dr = make_structs(d_in, d_out, tot_dev)
    # a stream of our own: the library takes a raw cudaStream_t (0 would select the engine's stream) and the
    # timing events must be recorded on the stream the kernels are launched on
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)

    kernel_ms = []
    score_ms = []

    # two engines, alternating: batch k+1 is queued while batch k runs; an engine is finished (its call waited
    # for, the tail kernels launched if any subject was handed on) before it is used again
    engines = [eng, g.engine((8 << 20) + 4096)]
    d_out2 = {k: torch.zeros(CAP[k] * SZ[k], dtype=torch.uint8, device=dev) for k in SZ}
    tot_dev2 = np.zeros(9, np.int64)
    _db2, dr2 = make_structs(d_in, d_out2, tot_dev2)
    results = [dr, dr2]
    in_flight = [False, False]
    turn = [0]

    def step_device_async():
        k = turn[0] & 1
        turn[0] += 1
        if in_flight[k]:
            _lib.check(lib.grimb_impute_finish(engines[k], C.byref(results[k])), "grimb_impute_finish")
        rc = lib.grimb_impute_device_async(engines[k], C.byref(cfg), C.byref(db), C.byref(results[k]),
                                           C.c_void_p(stream.cuda_stream))
        _lib.check(rc, "grimb_impute_device_async")
        in_flight[k] = True

    def finish_device():
        for k in (0, 1):
            if in_flight[k]:
                _lib.check(lib.grimb_impute_finish(engines[k], C.byref(results[k])), "grimb_impute_finish")
                in_flight[k] = False

    def step_device():
        rc = lib.grimb_impute_device(eng, C.byref(cfg), C.byref(db), C.byref(dr), C.c_void_p(stream.cuda_stream))
        _lib.check(rc, "grimb_impute_device")
        kernel_ms.append(lib.grimb_engine_kernel_ms(eng, 0))   # probe kernel, CUDA events inside the library
        score_ms.append(lib.grimb_engine_kernel_ms(eng, 4))    # k_fast_score (negative when the fused kernel runs)

    # host leg (pinned buffers; copies inside the timed region)
    h_in = {k: tens(as_signed(batch[k]), pin=True) for k in keys_in}
    h_out = {k: torch.zeros(CAP[k] * SZ[k], dtype=torch.uint8).pin_memory() for k in SZ}
    tot_host = np.zeros(9, np.int64)
    hb, hr = make_structs(h_in, h_out, tot_host)

    def step_host():
        rc = lib.grimb_impute_host(eng, C.byref(cfg), C.byref(hb), C.byref(hr))
        _lib.check(rc, "grimb_impute_host")

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup, drain=None):
        for _ in range(warmup):
            fn()
        if drain:
            drain()
        barrier()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
        ev[0].record(stream)
        for i in range(steps):
            fn()
            if drain and i == steps - 1:
                drain()          # every call of the timed region is complete (tails included) before its last event
            ev[i + 1].record(stream)
        barrier()
        ms = ev[0].elapsed_time(ev[steps])
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()) / steps

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = sum(lib.grimb_engine_launches(x) for x in engines)
    # `value`: back-to-back asynchronous calls (results and counters stay on the device until the end), so
    # the host turn-around between batches is hidden, as in a streaming caller
    ms_dev = timed(step_device_async, args.steps, args.warmup, drain=finish_device)
    last_out = None
    if args.dump_outputs and rank == 0:
        # the engines alternate, so the last timed call wrote the buffers of engine (turn - 1) & 1; the untimed
        # calls below reuse the first set
        bufs, tot = (d_out, tot_dev) if ((turn[0] - 1) & 1) == 0 else (d_out2, tot_dev2)
        last_out = (bufs["compact"].cpu().numpy().view(_lib.COMPACT_DTYPE),
                    bufs["words"][:int(tot[0]) * 8].cpu().numpy().view(np.uint64), int(tot[4]))
    launches = (sum(lib.grimb_engine_launches(x) for x in engines) - launches0) * args.steps // (args.steps + args.warmup)
    for _ in range(max(5, min(20, args.steps))):   # per-kernel device times: synchronous calls, events inside the library
        step_device()
    out_n = {"compact": S, "words": int(tot_dev[0]), "general": int(tot_dev[1]), "hap_rows": int(tot_dev[2]),
             "pop_rows": int(tot_dev[3])}
    evals = int(tot_dev[4])
    comp = d_out["compact"].cpu().numpy().view(_lib.COMPACT_DTYPE)
    status = comp["status"]
    gen = d_out["general"].cpu().numpy().view(_lib.SUBJECT_DTYPE)[:out_n["general"]]
    simple = (comp["kind_flags"] & 3) != 0
    # accepted phases (each = two haplotypes found in the table)
    hits = int((comp["kind_flags"][simple] >> 4).astype(np.int64).sum()) + int(gen["tot_pmug"].astype(np.int64).sum())
    ms_host = timed(step_host, args.steps, args.warmup)
    if rank == 0:
        # keep the GPU under the same load (untimed) until the clock sampler has a few readings
        t_end = time.time() + 4.0
        while len(sampler.rows) < 4 and time.time() < t_end:
            step_device()
    sampler.stop_flag = True

    # ---- spot parity against the oracle on the first subjects of rank 0 (not timed)
    parity = None
    cpu = None
    e2e_text = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:   # the CPU baseline is an N = 1 record
        import grim_oracle as go
        from grim.imputation.impute import Imputation
        n_c = min(S, args.cpu_sample)
        lines = subject_lines(names, alleles, 0, n_c)
        og = _FullOnlyGraph(names, fa, ff)
        oimp = go.OracleImputation(og, go.load_config(base_conf()), np.ones(1))
        t0 = time.time()
        ref = oimp.impute_lines(lines)
        t_cpu = time.time() - t0
        imp = Imputation(g, conf, np.ones(1))
        mine = {k: v.decode("utf8") for k, v in imp.impute_text("".join(lines).encode("utf8")).items()}
        parity = all(mine[k] == ref[k] for k in ref)
        # text in -> six texts out through grimb_impute_text (C++ tokeniser/formatter + kernels),
        # i.e. what grim.grim.impute(conf_file) does per chunk of the input file (not the headline)
        n_t = min(S, args.text_subjects)
        data = "".join(subject_lines(names, alleles, 0, n_t)).encode("utf8")
        imp.impute_text(data)           # warm-up at full size (pinned staging + device buffers grow once)
        imp2 = Imputation(g, conf, np.ones(1))
        imp2._text = imp._text
        t0 = time.time()
        texts = imp2.impute_text(data)
        t_text = time.time() - t0
        e2e_text = {"value": n_t / t_text, "unit": "subjects/s", "subjects": n_t, "in_bytes": len(data),
                    "out_bytes": sum(len(v) for v in texts.values()),
                    "tokenise_s": imp2.stats.get("tokenise_seconds"), "abi_s": imp2.stats.get("abi_seconds"),
                    "format_s": imp2.stats.get("format_seconds")}
        cpu = {"value": n_c / t_cpu, "unit": "subjects/s", "cores": 1, "kind": "port",
               "sample": "first %d of the %d subjects through oracle/grim_oracle.py on one core; outputs "
                         "compared with the CUDA path: %s" % (n_c, S, "identical" if parity else "DIFFERENT"),
               "pair_evals_per_sec": oimp.pair_evals / t_cpu}

    if rank == 0:
        total = S * world
        # algorithmic bytes (DESIGN.md "Measurement"): per subject its input (packed: 18 B = two keys + flags),
        # 2^L = 32 probes x one 32 B sector, per hit a 32 B frequency sector [the probe kernel];
        # the 16 B result record plus the words written [the score kernel].  The hand-over record between the
        # two is not counted.
        in_bytes_subject = sum(batch[k].nbytes for k in keys_in if k != "priors") / S
        out_bytes = sum(out_n[k] * SZ[k] for k in SZ)
        algo_probe = int(S * (in_bytes_subject + 32 * 32) + hits * 2 * 32)
        algo_path = algo_probe + out_bytes
        s_ms = [x for x in score_ms if x > 0]
        split = len(s_ms) > 0
        algo = algo_probe if split else algo_path   # the fused kernel (GRIMB_FAST_SPLIT=0) does both
        # for transparency: the probes the kernel really issues (homozygous loci collapse phases; SURVEY's
        # per-subject figure counts all 2^L side haplotypes, and that figure is what `achieved` uses)
        nhet = (alleles[:, :, 0] != alleles[:, :, 1]).sum(axis=1)
        probes_issued = float(np.where(nhet > 0, 2.0 ** nhet, 1.0).mean())
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        # dominant kernel: average device time of the timed launches (events recorded on the launch stream)
        k_ms = [x for x in kernel_ms if x > 0]
        ms_kernel = float(np.mean(k_ms)) if k_ms else ms_dev
        achieved = algo / (ms_kernel * 1e-3) / 1e9
        traffic = None   # DRAM bytes per launch from the committed ncu --set full capture of this kernel
        try:
            name = "r02_ncu_summary_k_fast_probe_final.txt" if split else "r01_ncu_summary_k_impute_fast_final.txt"
            txt = open(os.path.join(ROOT, "profiles", name)).read().splitlines()
            rd = [l for l in txt if l.startswith("dram__bytes_read.sum")][0].split()
            wr = [l for l in txt if l.startswith("dram__bytes_write.sum")][0].split()
            unit = {"Mbyte": 1e6, "Gbyte": 1e9, "Kbyte": 1e3, "byte": 1.0}
            traffic = float(rd[2]) * unit[rd[1]] + float(wr[2]) * unit[wr[1]]
        except Exception:
            pass
        # the probe-bound roofline (BASELINE north_star): what the memory system sustains for the probe's own
        # access shape -- independent random 32-byte sector loads over a table as large as the full-label
        # region -- measured by tools/sector_peak.cu on this pool's B200 (profiles/r01_sector_peak_b200.jsonl).
        # Sectors counted for the kernel: one per probe really issued plus one frequency sector per hit
        # (continuation sectors of longer chains are not counted, so the fraction is a lower bound).
        probe_bound = None
        try:
            mult = int(os.environ.get("GRIMB_FULL_LOAD_MULT", "8"))
            region = 16
            while region < 16 * mult * info.get("n_full", args.haps):
                region *= 2
            rows = [json.loads(l) for l in open(os.path.join(ROOT, "profiles", "r01_sector_peak_b200.jsonl"))]
            rows = [r for r in rows if r.get("kind") == "random_sector" and r["table_bytes"] >= region]
            size = min(r["table_bytes"] for r in rows)
            pk = max(r["gsectors_per_s"] for r in rows if r["table_bytes"] == size)
            sectors = S * probes_issued + hits * 2
            ach = sectors / (ms_kernel * 1e-3) / 1e9
            probe_bound = {"unit": "G sectors/s (32 B)", "achieved": ach, "peak": pk, "frac": ach / pk,
                           "sector_loads_per_launch": sectors, "full_label_region_bytes": region,
                           "peak_table_bytes": size,
                           "peak_source": "profiles/r01_sector_peak_b200.jsonl (tools/sector_peak.cu: random "
                                          "32-byte sector loads, 64 warps/SM, best of 1/2/4 loads in flight per thread)"}
        except Exception:
            pass
        h2d = sum(batch[k].nbytes for k in keys_in)
        d2h = out_bytes
        # what bounds e2e: the host link.  tools/pcie_peak.py measured, on this pool's B200 boxes, how long
        # the link alone needs for one step's bytes with both directions busy (profiles/r01_pcie_peak_b200.json)
        link = None
        try:
            pk = json.load(open(os.path.join(ROOT, "profiles", "r01_pcie_peak_b200.json")))
            floor_ms = pk["duplex_ms"] * max(h2d / pk["h2d_bytes"], d2h / pk["d2h_bytes"])
            link = {"bound": "pcie", "floor_ms_per_gpu_step": floor_ms, "frac": floor_ms / ms_host,
                    "d2h_alone_gbs": pk["d2h_alone_gbs"], "h2d_alone_gbs": pk["h2d_alone_gbs"],
                    "source": "profiles/r01_pcie_peak_b200.json (tools/pcie_peak.py: the same bytes, one pinned "
                              "copy per direction, both directions at once, no kernels)"}
        except Exception:
            pass
        line = {
            "metric": "subjects_per_sec", "value": total / (ms_dev * 1e-3), "unit": "subjects/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_dev, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(args),
            "pair_evals_per_sec": evals * world / (ms_dev * 1e-3),
            "e2e": {"value": total / (ms_host * 1e-3), "unit": "subjects/s", "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "ms_per_step": ms_host, "link": link,
                    # what the host's memory system / PCIe complex moves for the whole job (all ranks, both
                    # directions): the limiter of e2e scaling on one host (SCALE: 8 ranks share it)
                    "host_gbs_aggregate": (h2d + d2h) * world / (ms_host * 1e-3) / 1e9},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "peak_source": "MEASURED_PEAKS.json hbm_gbs (measured)" if peaks else "fallback",
                         "algorithmic_bytes_per_launch": algo, "probes_per_subject_counted": 32,
                         "probes_per_subject_issued": probes_issued,
                         "kernel": "k_fast_probe" if split else "k_impute_fast", "kernel_ms": ms_kernel,
                         "kernel_share_of_step": ms_kernel / ms_dev,
                         "probe_bound": probe_bound,
                         # the whole single-population path (probe + score kernels) against the same peak
                         "path": ({"kernels": "k_fast_probe + k_fast_score", "ms": ms_kernel + float(np.mean(s_ms)),
                                   "k_fast_score_ms": float(np.mean(s_ms)), "algorithmic_bytes": algo_path,
                                   "achieved": algo_path / ((ms_kernel + float(np.mean(s_ms))) * 1e-3) / 1e9,
                                   "frac": algo_path / ((ms_kernel + float(np.mean(s_ms))) * 1e-3) / 1e9 / peak}
                                  if split else None)},
            "cpu_baseline": cpu,
            "clocks": sampler.summary(),
            "table": {"n_nodes": info["n_nodes"], "device_bytes": info["device_bytes"], "build_s": t_build},
            "host": {"cpus": os.cpu_count(), "numa_bound_cpus_rank0": (len(numa_cpus) if numa_cpus else None)},
            "status_counts": {str(i): int(c) for i, c in enumerate(np.bincount(status, minlength=6)) if c},
            "handed_to_general_kernel": int(tot_dev[5]), "general_records": out_n["general"],
            "parity_sample_identical": parity,
            "e2e_text": e2e_text,
        }
        line["pair_evals_note"] = ("reference-equivalent count: iterations reaching impute.py:464 / :573 in the reference's "
                                   "schedule (rounds x candidates x output kinds), not operations the GPU performs")
        if world == 1 and not args.no_configs:
            # every other kernel of the path in the same run: C3 / C5 (k_impute_typed), C4 (k_impute), K0
            import bench_configs
            eng = None
            g.close()
            try:
                line["configs"] = bench_configs.run_all(args, names, fa, ff, torch, dev, stream, peak)
                line["configs"]["K0"]["C2_table"] = {"n_full": info["n_full"], "n_nodes": info["n_nodes"],
                                                     "device_bytes": info["device_bytes"], "build_s": t_build,
                                                     "note": "includes the host-side staging of bench.py's arrays"}
            except Exception as exc:   # the headline line must survive a failing sub-record
                line["configs"] = {"error": repr(exc)}
        if last_out is not None:
            dump_outputs(args.dump_outputs, *last_out)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
