"""Scratch probe (GPU): per-phase cycle counters for a workload/config."""
import sys, os, json
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__))); sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, 'tests'))
import numpy as np
import bench, dnab_testutil as util, dnastore_b200 as d
wl = sys.argv[1] if len(sys.argv) > 1 else 'cfg2'
n = int(sys.argv[2]) if len(sys.argv) > 2 else 15
cfg = ([int(x) for x in sys.argv[3:9]] + [0] * 6)[:6]  # cluster_size threads_per_cta t_columns table s_prev partition (0 = auto)
w = bench.WORKLOADS[wl]
m = util.machine_from_recipe(w['recipe']); c = m.compile(d.ErrorFlags(length=w['length'], global_=True))
dec = d.Decoder(c); dec.configure(cfg[0], cfg[1], cfg[2])
for key, v in zip(("table", "s_prev", "partition"), cfg[3:]):
    if v: dec.set_option(key, v)
reads = bench.make_reads(w, n, 7)
dec.viterbi(reads[:2])
dec.set_debug(True)
out = dec.viterbi(reads)
st = dec.stats(); dc = dec.debug_counters(); info = dec.info()
cols = max(dc['columns'], 1)
print(json.dumps(dict(fill_ms=round(st['last_fill_ms'],2), cfg=cfg, info=info, tb_ms=st['last_traceback_ms'], reads=n,
      per_column=dict(local_iters=dc['sweeps'] / cols, rounds=dc['rounds'] / cols, work_rank0=dc['work_rank0'] / cols, dirty_first=dc['dirty_first'] / cols, hops_t0=dc['hops_t0'] / cols, cyc_emit=dc['cyc_emit'] / cols,
                      cyc_closure=dc['cyc_closure'] / cols, cyc_pred=dc['cyc_pred'] / cols, **{k: dc[k] / cols for k in dc if k.startswith('cyc_') and k not in ('cyc_emit','cyc_closure','cyc_pred')}))))
