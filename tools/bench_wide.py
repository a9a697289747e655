#!/usr/bin/env python
"""Decoding rate on a machine with wide states (tests/test_gpu_wide_states.py, machine (d): a 1200-way selector composed
onto l4c4), on the read-batched kernel (kernel=1) and the push kernel (kernel=2).  Each rate is reads over the time of
whole dnab_viterbi_batch calls, taken with CUDA events, after one untimed call.  Also prints the side plane's bytes per
read (the high bytes of the wide states' records) and the card it ran on.
Usage: python tools/bench_wide.py [--reads N] [--steps K] [--out FILE]"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import dnastore_b200 as d  # noqa: E402
import test_gpu_wide_states as wide  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_wide.py measures on a CUDA device; none found")
    from benchdata import synth
    name = "d_selector_l4c4"
    compiled = wide._compiled(name)
    a = compiled.arrays()
    rng = np.random.default_rng(20261021)
    reads = []
    for _ in range(args.reads):
        seq, _ = wide._walk(a, rng)
        reads.append(synth.mutate(seq, rng, sub_rate=0.01, dup_rate=0.002, max_dup=2, del_rate=0.002, max_del=2).upper())
    lens = np.array([len(r) for r in reads])
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                          capture_output=True, text=True).stdout.strip()
    res = dict(machine=name, n_states=int(a["n_states"]), reads=len(reads), mean_len=float(lens.mean()),
               max_len=int(lens.max()), card=card, kernels={})
    n_wide = 0
    for kernel in (1, 2):
        dec = d.Decoder(compiled, device=0)
        dec.set_option("kernel", kernel)
        dec.viterbi(reads)  # warm-up: plan, tables, scratch
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        t0.record()
        for _ in range(args.steps):
            dec.viterbi(reads)
        t1.record()
        torch.cuda.synchronize()
        ms = t0.elapsed_time(t1) / args.steps
        if kernel == 1:
            n_wide = dec.batch_info()["wide_states"]  # (the same states are wide for both kernels)
        entry = dict(reads_per_s=len(reads) / (ms / 1e3), ms_per_call=ms, wide_states=n_wide,
                     side_plane_bytes_per_read=float((lens.max() + 1) * 2 * n_wide),
                     records_bytes_per_read=float((lens.max() + 1) * a["n_states"] * (a["k"] + 2)))
        if kernel == 1:
            entry["batch_info"] = {k: v for k, v in dec.batch_info().items()}
        else:
            entry["info"] = dec.info()
        res["kernels"][f"kernel={kernel}"] = entry
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
