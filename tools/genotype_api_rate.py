#!/usr/bin/env python
"""Rate of the device-resident genotype interface against the existing device route, on bench.py's workload
(C2: 2^20 fully typed 5-locus subjects, one population, the 1M-haplotype Zipf table).

  (a) device route: a pre-packed batch (bench.pack_batch) in HBM, grimb_impute_device, compact records only
  (b) genotype route: the [S][5][2] genotype tensor in HBM -> grimb_batch_from_genotypes -> grimb_impute_device
      -> grimb_results_rows -> row tensors in HBM (buffers allocated once, as a streaming caller would)
  (c) Imputation.impute_genotypes on the same CUDA tensor (the Python interface: buffer allocation, the workspace
      check and the results object included)

Each route is timed with CUDA events around `--steps` synchronous calls; the routes alternate `--runs` times.  Also
reported: the device times of grimb_batch_from_genotypes (grimb_engine_kernel_ms 7) and grimb_results_rows (8),
the probe and score kernels, and the card's name and power limit, read in the same process.

  python tools/genotype_api_rate.py [--subjects S] [--steps K] [--runs R] [--out FILE]"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "py-graph-imputation_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--subjects", type=int, default=1 << 20)
    ap.add_argument("--haps", type=int, default=1000000)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import bench
    from grim.imputation import _lib
    from grim.imputation.impute import Imputation
    from grim.imputation.networkx_graph import Graph
    from grim.run_impute_def import load_config

    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    names, fa, ff = bench.make_table(args.haps)
    conf = load_config(bench.base_conf())
    g = Graph(conf).from_arrays(names, fa, ff)
    lib = g.lib
    imp = Imputation(g, conf, np.ones(1))
    S = args.subjects
    _b, alleles = bench.make_subjects(fa, ff, S, bench.SUBJECT_SEED)
    eng = g.engine(imp.workspaces[0])
    stream = torch.cuda.Stream(dev)
    torch.cuda.set_stream(stream)
    sp = C.c_void_p(stream.cuda_stream)
    cfg = imp.cfg

    pk, pf = bench.pack_batch(alleles, g.key_bits, [len(a) for a in names])
    d_pk = torch.from_numpy(pk.view(np.int64)).to(dev)
    d_pf = torch.from_numpy(pf.view(np.int16)).to(dev)
    priors = torch.ones((1, 1, 1), dtype=torch.float64, device=dev)
    ids = torch.from_numpy(alleles).view(torch.int16).to(dev)
    packed = _lib.Batch()
    packed.n_subjects, packed.packed_keys, packed.packed_flags = S, d_pk.data_ptr(), d_pf.data_ptr()
    packed.priors, packed.n_priors = priors.data_ptr(), 1
    caps = (S * 2, S // 8 + 1024, S // 4 + 1024, S // 4 + 1024)
    out = [torch.zeros(c * sz, dtype=torch.uint8, device=dev) for c, sz in zip((S,) + caps, (16, 8, 48, 24, 16))]
    tot = np.zeros(9, np.int64)
    res = _lib.Results()
    res.compact, res.totals = out[0].data_ptr(), tot.ctypes.data
    res.words, res.word_capacity = out[1].data_ptr(), caps[0]
    res.general, res.general_capacity = out[2].data_ptr(), caps[1]
    res.hap_rows, res.hap_capacity = out[3].data_ptr(), caps[2]
    res.pop_rows, res.pop_capacity = out[4].data_ptr(), caps[3]
    # row buffers of (b): two rows per subject per kind is ample for this workload (checked after every call)
    L = 5
    rows = _lib.Rows()
    keep = {}
    for f, dt in (("status", torch.uint8), ("plan_umug", torch.uint8), ("plan_pmug", torch.uint8), ("flags", torch.uint8),
                  ("tot_umug", torch.int32), ("tot_pmug", torch.int32)):
        keep[f] = torch.empty(S, dtype=dt, device=dev)
        setattr(rows, f, keep[f].data_ptr())
    rcap = (S + 4096, 2 * S + 4096, S + 4096, S + 4096)
    for i, w in enumerate((2 * L, 2 * L, 2, 2)):
        keep["off%d" % i] = torch.empty(S + 1, dtype=torch.int64, device=dev)
        keep["rows%d" % i] = torch.empty(rcap[i] * w, dtype=torch.int16, device=dev)
        keep["prob%d" % i] = torch.empty(rcap[i], dtype=torch.float64, device=dev)
        rows.off[i], rows.rows[i], rows.prob[i] = keep["off%d" % i].data_ptr(), keep["rows%d" % i].data_ptr(), keep["prob%d" % i].data_ptr()
        rows.capacity[i] = rcap[i]
    rtot = np.zeros(4, np.int64)
    rows.totals = rtot.ctypes.data
    gb = _lib.Batch()

    def route_a():
        _lib.check(lib.grimb_impute_device(eng, C.byref(cfg), C.byref(packed), C.byref(res), sp), "grimb_impute_device", lib)

    def route_b():
        _lib.check(lib.grimb_batch_from_genotypes(eng, ids.data_ptr(), S, None, priors.data_ptr(), 1, None, C.byref(gb), sp),
                   "grimb_batch_from_genotypes", lib)
        _lib.check(lib.grimb_impute_device(eng, C.byref(cfg), C.byref(gb), C.byref(res), sp), "grimb_impute_device", lib)
        _lib.check(lib.grimb_results_rows(eng, C.byref(cfg), C.byref(gb), C.byref(res), C.byref(rows), sp),
                   "grimb_results_rows", lib)

    def route_c():
        imp.impute_genotypes(ids)

    def timed(fn):
        for _ in range(args.warmup):
            fn()
        stream.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(args.steps):
            fn()
        e1.record(stream)
        e1.synchronize()
        return e0.elapsed_time(e1) / args.steps

    result = {"gpu": gpu, "subjects": S, "table_haplotypes": args.haps, "steps": args.steps, "runs": []}
    for r in range(args.runs):
        run = {}
        for name, fn in (("a_device_route", route_a), ("b_genotype_route", route_b), ("c_impute_genotypes", route_c)):
            ms = timed(fn)
            run[name] = {"ms_per_batch": ms, "subjects_per_s": S / (ms * 1e-3)}
            if name == "b_genotype_route":
                run[name]["encode_ms_which7"] = lib.grimb_engine_kernel_ms(eng, 7)
                run[name]["rows_ms_which8"] = lib.grimb_engine_kernel_ms(eng, 8)
                run[name]["probe_ms_which0"] = lib.grimb_engine_kernel_ms(eng, 0)
                run[name]["score_ms_which4"] = lib.grimb_engine_kernel_ms(eng, 4)
                run[name]["probe_kernel_which6"] = lib.grimb_engine_kernel_ms(eng, 6)
                run[name]["rows"] = [int(x) for x in rtot]
            if name == "a_device_route":
                run[name]["probe_ms_which0"] = lib.grimb_engine_kernel_ms(eng, 0)
                run[name]["score_ms_which4"] = lib.grimb_engine_kernel_ms(eng, 4)
        run["b_over_a"] = run["b_genotype_route"]["subjects_per_s"] / run["a_device_route"]["subjects_per_s"]
        run["c_over_a"] = run["c_impute_genotypes"]["subjects_per_s"] / run["a_device_route"]["subjects_per_s"]
        result["runs"].append(run)
        print(json.dumps(run), flush=True)
    text = json.dumps(result, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")
    g.close()


if __name__ == "__main__":
    main()
