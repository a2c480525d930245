#!/usr/bin/env python
"""Rate of the device-resident route for ambiguous genotypes (Imputation.impute_genotype_lists:
grimb_batch_from_genotype_lists -> the imputation kernels -> grimb_results_rows) on C4-messy-shaped subjects
(synth.messy_subjects(table, N, 4, max_amb=6) on the README table).

  (1) device times of the last call's list encoder (grimb_engine_kernel_ms 9), k_impute (1) and row decode (8),
      from the CUDA events the library records (k_impute: its last launch; workspace_retries counts the subjects
      re-issued on a larger workspace tier, each re-issue a further launch; capacity_reruns counts the times the
      imputation ran again on larger result arrays)
  (2) the whole impute_genotype_lists call on CUDA tensors (host clock, ending in a device synchronise) against
      impute_text on the same lines (text in, six texts out)
  (3) a mixed batch, 80 % fully typed unambiguous subjects and 20 % ambiguous ones: impute_genotype_lists on the
      whole batch, and on its typed part alone, against impute_genotypes (the dense route) on the typed part

The measurements alternate `--runs` times in one process; the card's name and power limit are read in the same
process.

  python tools/genotype_lists_rate.py [--subjects N] [--runs R] [--out FILE]"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "py-graph-imputation_b200"), os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--subjects", type=int, default=100000)
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import goldenlib
    import synth
    from grim.imputation.impute import Imputation
    from grim.imputation.networkx_graph import Graph
    from grim.run_impute_def import load_config

    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    _t, conf, _l, _e = goldenlib.load_case("g1_readme_donor")
    cfg = load_config(conf)
    g = Graph(cfg).build_graph()
    imp = Imputation(g, cfg)
    dev = torch.device("cuda", g.device)
    eng = g.engine(imp.workspaces[0])
    tab = synth.Table(open(conf["freq_file"]).read())
    N = args.subjects

    def encode(lines):
        counts, alleles, _u, tp = imp.encode_genotype_lists([ln.rstrip().split(",")[1] for ln in lines])
        ok = np.setdiff1d(np.arange(len(lines)), tp)
        n = counts.astype(np.int64).sum((1, 2))
        off = np.concatenate([[0], np.cumsum(n)])
        sel = np.concatenate([np.arange(off[j], off[j + 1]) for j in ok] + [np.zeros(0, np.int64)])
        return ok, torch.from_numpy(counts[ok]).to(dev), torch.from_numpy(alleles[sel]).to(dev)

    messy = synth.messy_subjects(tab, N, 4, max_amb=6)
    ok, m_counts, m_alleles = encode(messy)
    m_text = "".join(messy[j] for j in ok).encode("utf8")
    n_typed = (N * 4) // 5
    typed = synth.typed_subjects(tab, n_typed, 5)
    amb = synth.messy_subjects(tab, N - n_typed, 6, max_amb=6)
    mixed = typed + amb
    _ok2, x_counts, x_alleles = encode(mixed)
    _ok3, t_counts, t_alleles = encode(typed)
    t_ids, _u, tp = imp.encode_genotypes([ln.rstrip().split(",")[1] for ln in typed])
    assert not tp
    t_ids = torch.from_numpy(t_ids).to(dev)

    def clock(fn):
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize(dev)
        return (time.perf_counter() - t0) * 1e3

    # warm every shape once
    imp.impute_genotype_lists(m_counts, m_alleles)
    imp.impute_text(m_text)
    imp.impute_genotype_lists(x_counts, x_alleles)
    imp.impute_genotype_lists(t_counts, t_alleles)
    imp.impute_genotypes(t_ids)
    result = {"gpu": gpu, "workload": "synth.messy_subjects(README table, %d, 4, max_amb=6)" % N,
              "subjects_taken": int(len(ok)), "alleles_listed": int(m_alleles.numel()),
              "mixed_batch": {"typed": n_typed, "ambiguous": N - n_typed}, "runs": []}
    for _r in range(args.runs):
        run = {}
        box = []
        ms = clock(lambda: box.append(imp.impute_genotype_lists(m_counts, m_alleles)))
        run["workspace_retries"] = box[0].workspace_retries
        run["capacity_reruns"] = box[0].capacity_reruns
        run["kernels_ms"] = {"list_encoder_which9": g.lib.grimb_engine_kernel_ms(eng, 9),
                             "k_impute_which1": g.lib.grimb_engine_kernel_ms(eng, 1),
                             "row_decode_which8": g.lib.grimb_engine_kernel_ms(eng, 8)}
        if run["workspace_retries"]:   # the re-issue's k_impute, on the next tier's engine
            run["kernels_ms"]["k_impute_which1_tier1"] = g.lib.grimb_engine_kernel_ms(g.engine(imp.workspaces[1]), 1)
        run["impute_genotype_lists_ms"] = ms
        run["impute_text_ms"] = clock(lambda: imp.impute_text(m_text))
        run["text_over_lists"] = run["impute_text_ms"] / ms
        run["mixed_lists_ms"] = clock(lambda: box.append(imp.impute_genotype_lists(x_counts, x_alleles)))
        run["mixed_capacity_reruns"] = box[-1].capacity_reruns
        run["typed_part_lists_ms"] = clock(lambda: imp.impute_genotype_lists(t_counts, t_alleles))
        run["typed_part_dense_ms"] = clock(lambda: imp.impute_genotypes(t_ids))
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
