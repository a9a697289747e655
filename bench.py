#!/usr/bin/env python
"""bench.py -- DP cells/s and decoded reads/s of the batched Viterbi decoder (--error-global).

Contract (see the task statement): `python bench.py --gpus N --steps K --warmup W` prints ONE JSON line on rank 0.
A "step" is one pass of the hot path (fill + traceback kernels) over ONE FIXED batch of synthetic reads, the same
total number of reads whatever N ("scaling": "strong"): reads are independent, so rank r decodes the r-th contiguous
shard of the batch (balanced by sum(L+1), dnastore_b200/sharding.py) with no collective on the data path, and the
decoded strings, log-likelihoods and statuses are gathered to rank 0 in input order INSIDE the timed region.

  value     whole-job DP cells/s, packed reads already resident in HBM (CUDA events on the launching stream,
            barrier + synchronize on both sides, max over ranks), ordered gather to rank 0 included
  e2e       the same batches through the product's own multi-GPU entry, dnab_viterbi_batch_multi (one process, one
            host thread and decoder per device, host buffers, H2D of reads and D2H of results inside the timed
            region, results in input order on the host); run by rank 0 over all N devices while the other ranks idle
  roofline  HBM roofline of the dominant kernel: algorithmic bytes = 1 B per DP cell + ceil(L/4) + |decoded| + 8
            per read (SURVEY.md 8d) / its CUDA-event time on rank 0
  cpu_baseline  (N = 1) the reference's own CPU decoder (oracle/_ref/dnastore) on a bounded sample of the same reads,
            one core; log-likelihood bits, traceback path and decoded string of every sampled read are compared with
            the GPU's through oracle/_ref/refdriver
  other_workloads  (N = 1) short runs of the other BASELINE machines and of forward-backward (reads/s, cells/s,
            roofline fraction, CPU reads/s), so that every configuration reaches the driver-run record

`--impl reference` times the UNMODIFIED reference CPU implementation (oracle/_ref, built from /root/reference by
oracle/Makefile) on all host cores, one process per core, same metric/config; it composes the machine with the
reference's own code (refdriver compose) and never imports this repository's library.

`--dump-outputs DIR` writes, after the timed steps, what the timed path returned for its last step as DIR/<name>.npy
(float64 stays float64, everything else becomes float32). The inputs depend only on the arguments, so two builds can
be compared output for output.
"""
import argparse
import atexit
import gzip
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

WORKLOADS = {
    # BASELINE.json configs[1]: the configuration the metric is quoted on
    "cfg2": dict(recipe=("l4c4", "flusher", "mixradar6"), pool="cfg2_flusher_mixradar6_l4c4_204b", length=4,
                 mut=dict(sub_rate=0.01), desc="flusher*mixradar6*dnastore-l4 (46,670 states), ~200-nt reads, 1% substitutions"),
    "cfg1": dict(recipe=("l4c4",), pool="cfg1_l4c4_200b", length=4, mut=dict(sub_rate=0.01),
                 desc="dnastore-l4 (384 states), ~200-nt reads, 1% substitutions"),
    "cfg3": dict(recipe=("l4c4", "sync16", "flusher", "hamming74"), pool="cfg3_s16h74l4c4_92b", length=4,
                 mut=dict(sub_rate=0.01, dup_rate=0.01, max_dup=2, del_rate=0.01, max_del=4),
                 desc="sync16*hamming74*dnastore-l4 (12,361 states), indels"),
    "cfg4": dict(recipe=("l4c4", "water64.1"), pool="cfg4_water64.1_l4c4_64b", length=4,
                 mut=dict(sub_rate=0.01, del_rate=0.01, max_del=4), desc="watermark64.1*dnastore-l4 (7,066 states)"),
    # BASELINE.json configs[4]'s machine (dnastore -l 8, 10,746 states, k = 4), 150-bit payloads, substitutions
    "cfg5": dict(recipe=("l8c4",), pool="cfg5_l8c4_150b", length=8, mut=dict(sub_rate=0.01),
                 desc="dnastore-l8 (10,746 states, k = 4), ~150-bit payloads, 1% substitutions"),
}
METRIC = "viterbi_dp_cells_per_sec"
UNIT = "cells/s"
# reads per step, the WHOLE job (fixed as N grows: strong scaling)
DEFAULT_BATCH = {"cfg2": 7680, "cfg1": 262144, "cfg3": 16384, "cfg4": 16384, "cfg5": 16384}


def make_reads(w, n, seed):
    from benchdata import synth
    pool = synth.load_pool(w["pool"])
    rng = np.random.default_rng(seed)
    base = [pool[i % len(pool)] for i in range(n)]
    mut = w["mut"]
    if set(mut) == {"sub_rate"}:
        return synth.mutate_subs_batch(base, rng, sub_rate=mut["sub_rate"])
    return [synth.mutate(s, rng, **mut) for s in base]


def cells_of(n_states, k, read_len):
    return int(n_states) * int(np.sum(np.asarray(read_len).astype(np.int64) + 1)) * (k + 2)


DUMP_BYTES = 60 << 20  # array data; with the .npy headers a dump stays under 64 MB (64e6 bytes)


def dump_outputs(directory, arrays):
    """--dump-outputs: arrays (name -> array whose first axis is the read / alignment) as <directory>/<name>.npy, plus
    index.npy, the row numbers written. All rows if they fit in DUMP_BYTES, else a fixed, seeded sample of rows."""
    n = len(next(iter(arrays.values())))
    out_dtype = {k: np.float64 if a.dtype == np.float64 else np.float32 for k, a in arrays.items()}
    row_bytes = 8 + sum(np.dtype(out_dtype[k]).itemsize * int(np.prod(a.shape[1:])) for k, a in arrays.items())
    m = min(n, DUMP_BYTES // row_bytes)
    index = np.arange(n) if m == n else np.sort(np.random.default_rng(0).choice(n, size=m, replace=False))
    os.makedirs(directory, exist_ok=True)
    np.save(os.path.join(directory, "index.npy"), index.astype(np.float64))
    for k, a in arrays.items():
        np.save(os.path.join(directory, k + ".npy"), a[index].astype(out_dtype[k]))


def decoded_matrix(strings):
    """Decoded strings as one byte code per symbol, zero-padded to the longest: [n, max length] uint8."""
    mat = np.zeros((len(strings), max((len(s) for s in strings), default=0)), dtype=np.uint8)
    for i, s in enumerate(strings):
        mat[i, :len(s)] = np.frombuffer(s.encode("latin1"), dtype=np.uint8)
    return mat


class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.device = device
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                                          "-i", str(self.device), "-lms", "200"], stdout=subprocess.PIPE, text=True)
            atexit.register(self.proc.kill)  # never outlive the benchmark, even when it fails before stop()
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _pump(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        self.proc.terminate()
        self.thread.join(timeout=2)
        sm, mx, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); power.append(float(f[3]))
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        if not sm:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["no samples"])
        return dict(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), reasons=sorted(reasons),
                    power_w_max=float(max(power)), samples=len(sm))


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ----------------------------------------------------------------------------------------------
# the reference's own CPU implementation (oracle/_ref): --impl reference and the cpu_baseline leg.
# Nothing in this section imports dnastore_b200.
# ----------------------------------------------------------------------------------------------
REF_BIN = os.path.join(ROOT, "oracle", "_ref", "dnastore")
REF_DRV = os.path.join(ROOT, "oracle", "_ref", "refdriver")
MACHINES = os.path.join(ROOT, "tests", "golden", "machines")


def ref_available():
    return all(os.path.exists(p) and os.access(p, os.X_OK) for p in (REF_BIN, REF_DRV))


def _gunzip_machine(name, keep):
    tf = tempfile.NamedTemporaryFile("wb", suffix=".json", delete=False)
    tf.write(gzip.open(os.path.join(MACHINES, name + ".json.gz"), "rb").read())
    tf.close()
    keep.append(tf.name)
    return tf.name


def ref_machine_json(w):
    """The workload's machine composed by the REFERENCE's own code (refdriver compose = Machine::compose), as a
    file; returns (path, n_states, k, temp files)."""
    temps = []
    base = _gunzip_machine(w["recipe"][0], temps)
    path = base
    if len(w["recipe"]) > 1:
        cmd = [REF_DRV, "compose", "--machine", base]
        for c in w["recipe"][1:]:
            cmd += ["--compose", _gunzip_machine(c, temps)]
        out = tempfile.NamedTemporaryFile("w", suffix=".json", delete=False)
        out.close()
        temps.append(out.name)
        subprocess.run(cmd + ["--save", out.name], check=True, capture_output=True)
        path = out.name
    text = open(path).read()
    try:
        states = json.loads(text)["state"]
        n_states = len(states)
        ctx = max((sum(1 for ch in st.get("l", "") if ch != "*") for st in states), default=0)
    except ValueError:  # the reference's writer is lenient about commas in places; count instead
        import re
        n_states = text.count('"n":')
        ctx = max((sum(1 for ch in m if ch != "*") for m in re.findall(r'"l":"([^"]*)"', text)), default=0)
    return path, n_states, min(ctx, w["length"] // 2), temps


def ref_cli_decode(w, machine_json, reads, n_procs):
    """`dnastore -v0 -l <len> --load-machine M -V shard.fa --error-global --raw` on n_procs cores, one process per
    core on disjoint shards; a machine-load-only run is subtracted (SURVEY.md 8d). Returns (seconds, decoded)."""
    shards = [s for s in (reads[i::n_procs] for i in range(n_procs)) if s]
    files = []
    for s in shards:
        tf = tempfile.NamedTemporaryFile("w", suffix=".fa", delete=False)
        for i, r in enumerate(s):
            tf.write(f">r{i}\n{r}\n")
        tf.close()
        files.append(tf.name)
    base = [REF_BIN, "-v0", "-l", str(w["length"]), "--load-machine", machine_json]
    t0 = time.perf_counter()
    subprocess.run(base + ["--save-machine", os.devnull], check=True, capture_output=True)
    t_load = time.perf_counter() - t0
    t0 = time.perf_counter()
    procs = [subprocess.Popen(base + ["-V", f, "--error-global", "--raw"] + list(w.get("ref_flags", [])), stdout=subprocess.PIPE, text=True)
             for f in files]
    outs = [p.communicate()[0] for p in procs]
    dt = time.perf_counter() - t0 - t_load
    for f in files:
        os.unlink(f)
    decoded = [None] * len(reads)
    for i, (o, s) in enumerate(zip(outs, shards)):
        decoded[i::n_procs] = o.split("\n")[:len(s)]
    return max(dt, 1e-9), decoded


def ref_driver_decode(w, machine_json, reads):
    """log-likelihood (hex float), decoded string and traceback path of every read from the reference's objects
    (refdriver viterbi: ViterbiMatrix::loglike / traceback). Untimed: this is the checker."""
    tf = tempfile.NamedTemporaryFile("w", suffix=".fa", delete=False)
    for i, r in enumerate(reads):
        tf.write(f">r{i}\n{r}\n")
    tf.close()
    flags = w.get("flags", {})
    cmd = [REF_DRV, "viterbi", "--machine", machine_json, "-l", str(w["length"]), "--sub", "0.01", "--iv", "10.0",
           "--dup", repr(flags.get("dup_prob", 0.001)), "--delopen", repr(flags.get("del_open", 0.001)), "--delext", "0.01",
           "--global", "--fasta", tf.name, "--path"]
    out = subprocess.run(cmd, check=True, capture_output=True, text=True).stdout
    os.unlink(tf.name)
    res = []
    for ln in out.split("\n"):
        if not ln:
            continue
        _name, _ll, llhex, decoded, pathstr = ln.split("\t")
        triples = [[int(x) for x in t.split(":")] for t in pathstr.split()] if pathstr else []
        res.append(dict(loglike_hex=llhex, decoded=decoded, path=triples[1:]))  # the start cell is logged twice
    return res


def reference_arm(args, w):
    """--impl reference: the unmodified reference on every host core, a bounded sample per step."""
    if not ref_available():
        print(json.dumps(dict(impl="reference", unavailable="oracle/_ref was not built (needs /root/reference at build time)")), flush=True)
        return
    mjson, n_states, k, temps = ref_machine_json(w)
    cores = os.cpu_count() or 1
    # calibration (untimed): one read per core, then as many reads per core as make a step of ~6 s
    cal = make_reads(w, cores, seed=999)
    dt_cal, _ = ref_cli_decode(w, mjson, cal, cores)
    per_core = int(min(512, max(1, round(6.0 / max(dt_cal, 1e-3)))))
    per_step = cores * per_core
    times, cells = [], []
    for step in range(args.warmup + args.steps):
        reads = make_reads(w, per_step, seed=1000 + step)
        dt, _dec = ref_cli_decode(w, mjson, reads, cores)
        if step >= args.warmup:
            times.append(dt)
            cells.append(cells_of(n_states, k, [len(r) for r in reads]))
    for t in temps:
        os.unlink(t)
    total_t = sum(times)
    value = sum(cells) / total_t
    ours = args.reads_per_step or DEFAULT_BATCH[args.workload]
    line = dict(impl="reference", metric=METRIC, value=value, unit=UNIT, n_gpus=args.gpus, steps=args.steps,
                warmup=args.warmup, ms_per_step=1e3 * total_t / max(args.steps, 1), higher_is_better=True,
                scaling="strong", vs_baseline=None, dtype="f64", data="synthetic",
                reads_per_sec=per_step * args.steps / total_t,
                config=dict(workload=f"{args.workload}: {w['desc']}, --error-global, -l {w['length']}",
                            reads_per_step=per_step, n_states=int(n_states), k=int(k),
                            note=f"a step of the GPU arm decodes {ours} reads; the CPU arm decodes {per_core} read(s) per core per step "
                                 f"(a bounded sample of the same distribution, sized for ~6 s per step: at 0.2-250 reads/s per core "
                                 f"the full batch would take hours) -- the metric is per DP cell, so the two are comparable",
                            machine="composed by the reference's own Machine::compose (oracle/_ref/refdriver compose)"),
                cpu_baseline=dict(value=value, unit=UNIT, cores=cores, kind="reference",
                                  sample=f"{per_step} reads per step ({per_core} per core), {args.steps} steps, oracle/_ref/dnastore -V"),
                e2e=dict(value=value, unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    print(json.dumps(line), flush=True)


def bench_fwdback(args, w, compiled, dec, rank, local_rank, world, dev, dist, torch, d, util):
    """Forward-backward step: dnab_fwdback_counts_batch over one batch of reads per GPU (host buffers; the
    copies are a few hundred bytes per read). Algorithmic bytes: 16 per DP cell (the forward cell is written
    once and read once by the backward pass, SURVEY.md 8d)."""
    t = compiled.t
    rps = args.reads_per_step or {"cfg5": 1184, "cfg1": 8192}.get(args.workload, 592)
    n_batches = args.warmup + args.steps
    batches = [make_reads(w, rps, seed=(rank + 1) * 200003 + b) for b in range(n_batches)]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for b in range(args.warmup):
        dec.fwdback_counts(batches[b])
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    barrier()
    kernel_ms, cells, max_gap = 0.0, 0, 0.0
    t0 = time.perf_counter()
    for b in range(args.warmup, n_batches):
        out = dec.fwdback_counts(batches[b])
        kernel_ms += dec.stats()["last_fill_ms"]  # CUDA events around the kernel, on its stream
        cells += cells_of(t.n_states, t.k, np.array([len(r) for r in batches[b]]))
        max_gap = max(max_gap, float(np.abs(out["loglike_back"] - out["loglike"]).max()))
        assert (out["status"] == 0).all()
    barrier()
    wall_s = time.perf_counter() - t0
    clocks = sampler.stop() if rank == 0 else None
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, out)
    vals = torch.tensor([kernel_ms, wall_s], dtype=torch.float64, device=dev)
    sums = torch.tensor([float(cells), float(rps * args.steps)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(vals, op=dist.ReduceOp.MAX)
        dist.all_reduce(sums, op=dist.ReduceOp.SUM)
    kernel_ms_max, wall_max = vals.tolist()
    tot_cells, tot_reads = sums.tolist()
    if rank == 0:
        peak, peak_src = measured_peak()
        achieved = 16.0 * cells / (kernel_ms * 1e-3) / 1e9
        cpu = None
        if args.cpu_sample > 0:
            sample = batches[-1][:min(args.cpu_sample, 2)]
            t1 = time.perf_counter()
            ref = [util.oracle_fwdback(compiled, r) for r in sample]
            dt = time.perf_counter() - t1
            for i, o in enumerate(ref):
                assert util.hexf(o["loglike"]) == util.hexf(out["loglike"][i]), "GPU forward log-likelihood differs from the specification"
                np.testing.assert_allclose(out["counts"][i], o["counts"], rtol=1e-9, atol=1e-12)
            cpu_cells = cells_of(t.n_states, t.k, np.array([len(r) for r in sample]))
            cpu = dict(value=cpu_cells / dt, unit=UNIT, cores=1, kind="port", reads_per_sec=len(sample) / dt,
                       sample=f"first {len(sample)} reads of the last timed batch through oracle/forward_oracle.c (a specification: "
                              f"the reference has no machine-lattice forward-backward), results equal to the GPU's; host has {os.cpu_count()} cores")
        line = dict(metric="fwdback_dp_cells_per_sec", value=tot_cells / (kernel_ms_max * 1e-3), unit=UNIT, n_gpus=world,
                    steps=args.steps, warmup=args.warmup, ms_per_step=1e3 * wall_max / args.steps, higher_is_better=True,
                    scaling="weak", vs_baseline=None, dtype="f64", data="synthetic",
                    reads_per_sec=tot_reads / (kernel_ms_max * 1e-3),
                    config=dict(workload=f"{args.workload}: {w['desc']}, --error-global, -l {w['length']}; forward + backward + "
                                         "posterior counts (parity unpinned: not in the reference)",
                                reads_per_step_per_gpu=rps, n_states=int(t.n_states), k=int(t.k),
                                l2="distinct read batch per step; the forward cells (8 B each) are streamed to HBM and read back",
                                max_abs_loglike_back_minus_forward=max_gap),
                    e2e=dict(value=tot_cells / wall_max, unit=UNIT, h2d_bytes_per_step=int(sum((len(r) + 3) // 4 + 12 for r in batches[-1])),
                             d2h_bytes_per_step=int(rps * (8 * (5 + t.k + 16) + 20)), steps=args.steps,
                             reads_per_sec=tot_reads / wall_max),
                    gpu_launches=int(args.steps * world),
                    roofline=dict(bound="hbm", achieved=achieved, peak=peak, unit="GB/s", frac=achieved / peak, traffic=None,
                                  kernel="forwardKernel", launches=args.steps, avg_launch_ms=kernel_ms / args.steps,
                                  peak_source=peak_src, algorithmic_bytes_per_launch=16.0 * cells / args.steps),
                    cpu_baseline=cpu, clocks=clocks)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


# ----------------------------------------------------------------------------------------------
def short_run(d, util, torch, dev, name, n_reads, steps=2, cpu_reads=2):
    """other_workloads: a short device-resident run of one more BASELINE machine on this GPU."""
    w = WORKLOADS[name]
    machine = util.machine_from_recipe(w["recipe"])
    compiled = machine.compile(d.ErrorFlags(length=w["length"], global_=True))
    t = compiled.t
    dec = d.Decoder(compiled, device=dev.index)
    binfo = dec.batch_info()
    batches = [d.pack_reads(make_reads(w, n_reads, seed=555 + b)) for b in range(steps + 1)]
    max_len = max(int(b[2].max()) for b in batches)
    stride = 2 * max_len + 64
    devb = [tuple(torch.from_numpy(a).to(dev) for a in b) for b in batches]
    o_ll = torch.zeros(n_reads, dtype=torch.float64, device=dev)
    o_dec = torch.zeros(n_reads * stride, dtype=torch.uint8, device=dev)
    o_len = torch.zeros(n_reads, dtype=torch.int32, device=dev)
    o_st = torch.zeros(n_reads, dtype=torch.int32, device=dev)
    stream = torch.cuda.current_stream().cuda_stream

    def run(b):
        p, o, l = devb[b]
        dec.viterbi_device(n_reads, max_len, p.data_ptr(), o.data_ptr(), l.data_ptr(), o_ll.data_ptr(), o_dec.data_ptr(), stride,
                           o_len.data_ptr(), o_st.data_ptr(), stream)
    run(0)
    torch.cuda.synchronize()
    dec.set_timing(True)
    dec.reset_timing()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for b in range(1, steps + 1):
        run(b)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    st = dec.stats()
    cells = sum(cells_of(t.n_states, t.k, batches[b][2]) for b in range(1, steps + 1))
    peak, _ = measured_peak()
    algo = cells + sum(int(np.sum((batches[b][2].astype(np.int64) + 3) // 4)) + 8 * n_reads for b in range(1, steps + 1)) \
        + int(o_len.sum().item()) * steps
    out = dict(workload=f"{name}: {w['desc']}", n_states=int(t.n_states), k=int(t.k), reads_per_step=n_reads, steps=steps,
               kernel="viterbiFillBatchKernel" if binfo["enabled"] else "viterbiFillPushKernel",
               reads_per_sec=n_reads * steps / (ms * 1e-3), cells_per_sec=cells / (ms * 1e-3),
               roofline_frac=algo / (st["timed_fill_ms"] * 1e-3) / 1e9 / peak, all_status_ok=bool((o_st == 0).all().item()))
    if cpu_reads and ref_available():
        mjson, _n, _k, temps = ref_machine_json(w)
        reads = make_reads(w, cpu_reads, seed=555 + steps)
        dt, cpu_dec = ref_cli_decode(w, mjson, reads, 1)
        gpu = dec.viterbi(reads)
        assert cpu_dec == gpu["decoded"], f"{name}: GPU decoded strings differ from the reference CLI's"
        out["cpu_reads_per_sec_one_core"] = cpu_reads / dt
        for tmp in temps:
            os.unlink(tmp)
    return out


def short_fwdback(d, util, n_reads=296):
    w = WORKLOADS["cfg5"]
    compiled = util.machine_from_recipe(w["recipe"]).compile(d.ErrorFlags(length=w["length"], global_=True))
    t = compiled.t
    dec = d.Decoder(compiled, device=0)
    reads = make_reads(w, n_reads, seed=901)
    dec.fwdback_counts(reads[:32])
    out = dec.fwdback_counts(reads)
    ms = dec.stats()["last_fill_ms"]
    cells = cells_of(t.n_states, t.k, [len(r) for r in reads])
    peak, _ = measured_peak()
    return dict(workload=f"cfg5 forward + backward + posterior counts (parity unpinned: not in the reference): {w['desc']}",
                reads_per_step=n_reads, reads_per_sec=n_reads / (ms * 1e-3), cells_per_sec=cells / (ms * 1e-3),
                roofline_frac=16.0 * cells / (ms * 1e-3) / 1e9 / peak, kernel="forwardKernel",
                max_abs_loglike_back_minus_forward=float(np.abs(out["loglike_back"] - out["loglike"]).max()))


def short_pairhmm(d, n_distinct=8192, copies=16, seed=77, steps=1, warmup=1, dump=None):
    """Batched pair-HMM forward + backward + expected counts (SURVEY.md 8a-11 / 8f-2) on synthetic alignments:
    reference-encoded ~200-nt strands mutated by the errdecode.pl simulator with the alignment kept
    (benchdata/synth.mutate_aligned), n_distinct alignments repeated `copies` times (the kernel deals alignments to warps in
    order of length, so a warp of 32 holds at least 32 / copies different alignments). DP cells = envelope cells x (2 + k);
    16 algorithmic bytes per DP cell (the forward cell is written once and read once by the counts pass). `warmup`
    untimed calls on the distinct alignments, then `steps` timed calls on the whole batch."""
    from benchdata import synth
    rng = np.random.default_rng(seed)
    pool = synth.load_pool("cfg1_l4c4_200b")
    rows = []
    for i in range(n_distinct):
        a, b = synth.mutate_aligned(pool[i % len(pool)], rng, sub_rate=0.02, dup_rate=0.01, max_dup=3, del_rate=0.01, max_del=4)
        rows.append(f"# STOCKHOLM 1.0\nin  {a}\nout {b}\n//\n")
    tf = tempfile.NamedTemporaryFile("w", suffix=".stk", delete=False)
    tf.write("".join(rows))
    tf.close()
    db = d.PairDb(tf.name)
    os.unlink(tf.name)
    params = d.MutatorParams.from_flags(d.ErrorFlags(length=12, sub_prob=.02, dup_prob=.01, del_open=.01, del_ext=.3))
    base = [db.alignment(i) for i in range(len(db))]
    aligns = base * copies
    k = params.max_dup_len
    cells = 0
    for tin, tout, ea, eb in base:
        cells += int((np.abs(ea[:, None] - eb[None, :]) <= k).sum())
    cells *= copies * (2 + k)
    for _ in range(warmup):
        d.pairhmm_fb_batch(params, base, strict=False)
    ms = 0.0  # mean kernel time of a timed call
    for _ in range(steps):
        fwd, back, counts, step_ms = d.pairhmm_fb_batch(params, aligns, strict=False)
        ms += step_ms / steps
    if dump:
        dump_outputs(dump, dict(fwd=fwd, back=back, counts=np.array([c.flat() for c in counts])))
    peak, _ = measured_peak()
    return dict(workload=f"pair-HMM forward + backward + expected counts, {len(aligns)} alignments ({len(base)} distinct) of ~200-nt strands, k = {k}, banded envelope",
                alignments=len(aligns), steps=steps, dp_cells=cells, kernel_ms=ms, alignments_per_sec=len(aligns) / (ms * 1e-3),
                cells_per_sec=cells / (ms * 1e-3), roofline_frac=16.0 * cells / (ms * 1e-3) / 1e9 / peak, kernel="pairHmmFwdBackKernel",
                max_abs_back_minus_fwd=float(np.abs(np.asarray(fwd) - np.asarray(back)).max()))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg2", choices=sorted(WORKLOADS))
    ap.add_argument("--reads-per-step", type=int, default=0, help="reads per step, whole job (0 = default for the workload)")
    ap.add_argument("--opt", action="append", default=[], help="decoder option key=value (dnab_decoder_set_option), repeatable")
    ap.add_argument("--cpu-sample", type=int, default=4, help="reads in the single-core CPU baseline sample (0 = skip)")
    ap.add_argument("--others", type=int, default=-1, help="other_workloads: 1 on, 0 off, -1 = on for N = 1 and the default workload")
    ap.add_argument("--no-indel", action="store_true", help="decode with --error-del-open 0 --error-dup-prob 0 (closure degenerates)")
    ap.add_argument("--mode", default="viterbi", choices=["viterbi", "fwdback", "pairhmm"],
                    help="fwdback: forward + backward + posterior counts over the machine lattice (weak scaling, one batch per GPU)")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    w = WORKLOADS[args.workload]
    if args.no_indel:
        # SURVEY.md 8d: the same workload decoded with --error-del-open 0 --error-dup-prob 0 -- the within-column
        # closure degenerates to one visit per state, an upper bound on what the exact closure costs
        w = dict(w, flags=dict(del_open=0., dup_prob=0.), ref_flags=["--error-del-open", "0", "--error-dup-prob", "0"],
                 desc=w["desc"] + ", --error-del-open 0 --error-dup-prob 0")

    if args.impl == "reference":
        if rank == 0:
            reference_arm(args, w)
        return

    import __graft_entry__ as g
    if rank == 0:
        g.build()
    if args.mode == "pairhmm":
        if rank == 0:
            import dnastore_b200 as d
            print(json.dumps(short_pairhmm(d, copies=max(1, args.reads_per_step // 8192) if args.reads_per_step else 16,
                                           steps=args.steps, warmup=args.warmup, dump=args.dump_outputs)), flush=True)
        return
    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    host_group = None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        dist.barrier()
        host_group = dist.new_group(backend="gloo")  # host-side waits that leave no kernel spinning on an idle GPU
    dev = torch.device("cuda", local_rank)
    import dnab_testutil as util
    import dnastore_b200 as d
    from dnastore_b200 import sharding

    machine = util.machine_from_recipe(w["recipe"])
    compiled = machine.compile(d.ErrorFlags(length=w["length"], global_=True, **w.get("flags", {})))
    t = compiled.t
    dec = d.Decoder(compiled, device=local_rank)
    for kv in args.opt:
        key, value = kv.split("=")
        dec.set_option(key, int(value))
    if args.mode == "fwdback":
        return bench_fwdback(args, w, compiled, dec, rank, local_rank, world, dev, dist, torch, d, util)
    binfo = dec.batch_info()
    info = dec.info() if not binfo["enabled"] else None
    total = args.reads_per_step or DEFAULT_BATCH[args.workload]

    # ---- the fixed batches (identical on every rank), this rank's contiguous shard resident in HBM -----------
    n_batches = args.warmup + args.steps
    full = []      # (reads of the last batch or None, packed, byte_off, read_len) of the WHOLE batch: rank 0's e2e leg
    mine = []      # this rank's shard, packed on its own
    bounds = []
    for b in range(n_batches):
        reads = make_reads(w, total, seed=100003 + b)
        lens = np.array([len(r) for r in reads], dtype=np.int64)
        cuts = sharding.shard_bounds(lens, world)
        bounds.append(cuts)
        lo, hi = int(cuts[rank]), int(cuts[rank + 1])
        mine.append(d.pack_reads(reads[lo:hi]))
        if rank == 0:
            full.append((reads if b == n_batches - 1 else None,) + tuple(d.pack_reads(reads)))
        else:
            full.append((None, None, None, lens.astype(np.int32)))
    max_len = max(int(f[3].max()) for f in full)
    stride = 2 * max_len + 64  # decoded strings are ~1 symbol per base for these codes
    shard_max = max(int(c[r + 1] - c[r]) for c in bounds for r in range(world))

    def to_dev(a):
        return torch.from_numpy(a).to(dev)

    dev_batches = [tuple(to_dev(a) for a in m) for m in mine]
    # results of this rank's shard; rank 0 also holds the gathered whole (fixed-size slots per rank)
    d_ll = torch.zeros(shard_max, dtype=torch.float64, device=dev)
    d_dec = torch.zeros(shard_max * stride, dtype=torch.uint8, device=dev)
    d_meta = torch.zeros(2 * shard_max, dtype=torch.int32, device=dev)  # decoded_len | status
    g_ll = [torch.zeros_like(d_ll) for _ in range(world)] if (rank == 0 and world > 1) else None
    g_dec = [torch.zeros_like(d_dec) for _ in range(world)] if (rank == 0 and world > 1) else None
    g_meta = [torch.zeros_like(d_meta) for _ in range(world)] if (rank == 0 and world > 1) else None
    stream = torch.cuda.current_stream().cuda_stream

    def run_device(b):
        p, o, l = dev_batches[b]
        n = int(l.numel())
        if n:
            dec.viterbi_device(n, max_len, p.data_ptr(), o.data_ptr(), l.data_ptr(), d_ll.data_ptr(), d_dec.data_ptr(), stride,
                               d_meta.data_ptr(), d_meta.data_ptr() + 4 * shard_max, stream)
        if world > 1:  # ordered gather: contiguous shards in rank order = input order
            dist.gather(d_ll, g_ll, dst=0)
            dist.gather(d_dec, g_dec, dst=0)
            dist.gather(d_meta, g_meta, dst=0)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for b in range(args.warmup):
        run_device(b)
    barrier()
    dec.set_timing(True)
    dec.reset_timing()
    launches0 = dec.stats()["kernel_launches"]
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    for b in range(args.warmup, n_batches):
        run_device(b)
    ev1.record()
    barrier()
    elapsed_ms = ev0.elapsed_time(ev1)
    st = dec.stats()
    dec.set_timing(False)
    clocks = sampler.stop() if rank == 0 else None
    gpu_launches = int(st["kernel_launches"] - launches0)
    n_mine_last = int(dev_batches[-1][2].numel())
    status_ok = bool((d_meta[shard_max:shard_max + n_mine_last] == 0).all().item())
    my_dec_bytes = int(d_meta[:n_mine_last].sum().item())
    my_cells = sum(cells_of(t.n_states, t.k, mine[b][2]) for b in range(args.warmup, n_batches))
    my_reads = sum(len(mine[b][2]) for b in range(args.warmup, n_batches))
    # what rank 0 holds after the last gather, in input order (checked against the e2e leg and the CPU below)
    gathered_dec, gathered_ll = None, None
    if rank == 0:
        cuts = bounds[-1]
        parts_ll = g_ll if world > 1 else [d_ll]
        parts_dec = g_dec if world > 1 else [d_dec]
        parts_meta = g_meta if world > 1 else [d_meta]
        gathered_dec, gathered_ll, gathered_status = [], [], []
        for r in range(world):
            n_r = int(cuts[r + 1] - cuts[r])
            ll = parts_ll[r][:n_r].cpu().numpy()
            dl = parts_meta[r][:n_r].cpu().numpy()
            raw = parts_dec[r][:n_r * stride].cpu().numpy().reshape(n_r, stride)
            gathered_ll.extend(ll.tolist())
            gathered_dec.extend(bytes(raw[i, :dl[i]]).decode("latin1") for i in range(n_r))
            gathered_status.extend(parts_meta[r][shard_max:shard_max + n_r].cpu().numpy().tolist())
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, dict(loglike=np.array(gathered_ll, dtype=np.float64), status=np.array(gathered_status),
                                                 decoded_len=np.array([len(s) for s in gathered_dec]),
                                                 decoded=decoded_matrix(gathered_dec)))

    # ---- e2e: the product's multi-GPU entry on rank 0 over all N devices, host buffers, every step ---------------
    del dev_batches
    e2e_s, e2e_h2d, e2e_d2h, e2e_ok = 0.0, 0, 0, True
    dec = None
    torch.cuda.empty_cache()
    barrier()

    def host_barrier():  # the other ranks' GPUs must be idle while rank 0 drives them: wait on the host (gloo), not in a NCCL kernel
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier(group=host_group)
    host_barrier()
    if rank == 0:
        md = d.MultiDecoder(compiled, list(range(world)))
        for kv in args.opt:
            key, value = kv.split("=")
            md.set_option(key, int(value))

        def pin(a):
            return torch.from_numpy(a).pin_memory().numpy()
        host = [(pin(f[1]), pin(f[2]), pin(f[3])) for f in full]
        out = dict(loglike=pin(np.zeros(total, dtype=np.float64)), raw=pin(np.zeros((total, stride), dtype=np.uint8)),
                   decoded_len=pin(np.zeros(total, dtype=np.int32)), status=pin(np.zeros(total, dtype=np.int32)))
        md.viterbi_packed(*host[0], decoded_stride=stride, out=out)  # warm the staging buffers of every device
        t0 = time.perf_counter()
        for b in range(args.warmup, n_batches):
            md.viterbi_packed(*host[b], decoded_stride=stride, out=out)
        e2e_s = time.perf_counter() - t0
        e2e_h2d = int(np.mean([h[0].nbytes + h[1].nbytes + h[2].nbytes for h in host[args.warmup:]]))
        e2e_d2h = int(out["loglike"].nbytes + out["raw"].nbytes + out["decoded_len"].nbytes + out["status"].nbytes)
        e2e_ok = out["decoded"] == gathered_dec and out["loglike"].tolist() == gathered_ll and bool((out["status"] == 0).all())
        assert e2e_ok, "the multi-GPU entry and the sharded device path disagree"
        md = None
    host_barrier()

    # ---- reduce over ranks: max time, summed work -------------------------------------------------------
    vals = torch.tensor([elapsed_ms, st["timed_fill_ms"], st["timed_traceback_ms"]], dtype=torch.float64, device=dev)
    sums = torch.tensor([my_cells, my_reads, float(gpu_launches), float(status_ok)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(vals, op=dist.ReduceOp.MAX)
        dist.all_reduce(sums, op=dist.ReduceOp.SUM)
    elapsed_ms, fill_ms, tb_ms = vals.tolist()
    tot_cells, tot_reads, tot_launches, n_ok = sums.tolist()

    if rank == 0:
        peak, peak_src = measured_peak()
        # roofline of the fill kernel on rank 0 (per launch)
        fl = max(int(st["timed_fill_launches"]), 1)
        algo_bytes = my_cells + sum(int(np.sum((mine[b][2].astype(np.int64) + 3) // 4)) for b in range(args.warmup, n_batches)) \
            + my_dec_bytes * args.steps + 8 * my_reads
        achieved = algo_bytes / (st["timed_fill_ms"] * 1e-3) / 1e9
        fill_kernel = "viterbiFillBatchKernel" if binfo["enabled"] else "viterbiFillPushKernel"
        traffic, traffic_src = None, None
        tp = os.path.join(ROOT, "profiles", "r02_fill_traffic.json")
        if os.path.exists(tp):
            tj = json.load(open(tp)).get(args.workload)
            if tj and tj.get("kernel") == fill_kernel:
                traffic = tj["dram_over_algorithmic"] * algo_bytes / fl
                traffic_src = tj["capture"]
        # CPU baseline (N = 1): the reference CLI on one core, timed; every sampled read's log-likelihood bits,
        # traceback path and decoded string compared with the GPU's through refdriver
        cpu = None
        if args.cpu_sample > 0 and world == 1 and ref_available():
            sample = full[-1][0][:args.cpu_sample]
            mjson, _n, _k, temps = ref_machine_json(w)
            dt, cpu_dec = ref_cli_decode(w, mjson, sample, 1)
            ref = ref_driver_decode(w, mjson, sample)
            chk = d.Decoder(compiled, device=0)
            for kv in args.opt:
                key, value = kv.split("=")
                chk.set_option(key, int(value))
            got = chk.viterbi(sample, want_path=True)
            for i, r in enumerate(ref):
                assert cpu_dec[i] == r["decoded"] == got["decoded"][i] == gathered_dec[i], f"read {i}: decoded strings differ from the reference"
                assert util.hexf(r["loglike_hex"]) == util.hexf(got["loglike"][i]) == util.hexf(gathered_ll[i]), \
                    f"read {i}: log-likelihood bits differ from the reference"
                assert got["path"][i].tolist() == r["path"], f"read {i}: traceback path differs from the reference"
            for tmp in temps:
                os.unlink(tmp)
            cpu_cells = cells_of(t.n_states, t.k, [len(r) for r in sample])
            cpu = dict(value=cpu_cells / dt, unit=UNIT, cores=1, kind="reference", reads_per_sec=len(sample) / dt,
                       sample=f"first {len(sample)} reads of the last timed batch, oracle/_ref/dnastore -V on one core; log-likelihood "
                              f"bits, traceback paths and decoded strings identical to the GPU's; host has {os.cpu_count()} cores")
        others = None
        want_others = args.others == 1 or (args.others == -1 and world == 1 and args.workload == "cfg2" and not args.opt)
        if want_others:
            others = {}
            for name, n in (("cfg1", 65536), ("cfg3", 2048), ("cfg4", 4096), ("cfg5", 4096)):
                if name != args.workload:
                    others[name] = short_run(d, util, torch, dev, name, n)
            others["cfg5_fwdback"] = short_fwdback(d, util)
            others["pairhmm"] = short_pairhmm(d)
        kernel_cfg = (dict(kernel="read-batched (viterbi_fill_batch.cu): 32 reads per group are the SIMD lanes",
                           team_size=binfo["team_size"], states_per_cta=binfo["states_per_cta"],
                           threads_per_cta=32 * binfo["warps_per_cta"], smem_bytes_per_cta=binfo["smem_bytes_per_cta"],
                           reads_in_flight=32 * binfo["n_teams"],
                           cross_cta_transition_fraction=round(binfo["cross_cta_transition_fraction"], 4))
                      if binfo["enabled"] else
                      dict(kernel="one read per cluster (viterbi_fill_push.cu)",
                           cluster_size=info["cluster_size"], states_per_cta=info["states_per_cta"],
                           threads_per_cta=info["threads_per_cta"], smem_bytes_per_cta=info["smem_bytes_per_cta"],
                           t_in_smem=info["t_in_smem"], table_in_smem=info["table_in_smem"], reads_in_flight=info["n_clusters"]))
        line = dict(
            metric=METRIC, value=tot_cells / (elapsed_ms * 1e-3), unit=UNIT, n_gpus=world, steps=args.steps,
            warmup=args.warmup, ms_per_step=elapsed_ms / args.steps, higher_is_better=True, scaling="strong",
            vs_baseline=None, dtype="f64", data="synthetic",
            reads_per_sec=tot_reads / (elapsed_ms * 1e-3),
            config=dict(workload=f"{args.workload}: {w['desc']}, --error-global, -l {w['length']}",
                        reads_per_step=total, shards="contiguous, balanced by sum(L+1), one per rank; results gathered to rank 0 "
                        "in input order inside the timed region (NCCL gather of fixed-size slots)" if world > 1 else "one GPU",
                        n_states=int(t.n_states), k=int(t.k), **kernel_cfg,
                        l2="a distinct batch per step; every step streams reads_per_step x (L+1) x n_states x (k+2) bytes of "
                           "predecessor records (>> L2)",
                        all_status_ok=bool(n_ok == world)),
            e2e=dict(value=tot_cells / e2e_s, unit=UNIT, h2d_bytes_per_step=e2e_h2d, d2h_bytes_per_step=e2e_d2h,
                     steps=args.steps, reads_per_sec=tot_reads / e2e_s,
                     path=f"dnab_viterbi_batch_multi over {world} device(s): one process, one host thread and decoder per "
                          "device, pinned host buffers in and out, results in input order; equal to the gathered results"),
            gpu_launches=int(tot_launches),
            roofline=dict(bound="hbm", achieved=achieved, peak=peak, unit="GB/s", frac=achieved / peak,
                          traffic=traffic, traffic_source=traffic_src,
                          kernel=fill_kernel, launches=fl, avg_launch_ms=st["timed_fill_ms"] / fl,
                          peak_source=peak_src, algorithmic_bytes_per_launch=algo_bytes / fl,
                          fill_share_of_step=fill_ms / elapsed_ms, traceback_share_of_step=tb_ms / elapsed_ms),
            cpu_baseline=cpu, other_workloads=others, clocks=clocks)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    sys.dont_write_bytecode = True  # the tree may be read-only; the benchmark writes nothing there
    main()
