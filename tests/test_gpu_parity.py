"""GPU (B200): the CUDA path, called through the C ABI, against the golden vectors made by
the unmodified reference and against the oracle on the same seeded inputs.

Bar: bit-exact fp64 log-likelihoods, identical decoded strings, identical traceback
paths, identical DP cells.
"""
import json

import numpy as np
import pytest

import dnab_testutil as util

pytestmark = pytest.mark.gpu

CASES = [c["name"] for c in util.load_golden()]


@pytest.fixture(scope="module")
def d():
    import dnastore_b200
    return dnastore_b200


def _check_against_golden(d, case, configure=None, options=None):
    compiled = util.compiled_for_case(case)
    dec = d.Decoder(compiled, device=0)
    if configure:
        dec.configure(**configure)
    for key, value in (options or {}).items():
        dec.set_option(key, value)
    reads = [r["seq"] for r in case["reads"]]
    out = dec.viterbi(reads, want_path=True)
    for i, r in enumerate(case["reads"]):
        tag = (case["name"], r["name"], configure)
        assert out["decoded"][i] == r["decoded"], tag
        assert util.hexf(out["loglike"][i]) == util.hexf(r["loglike_hex"]), tag
        assert out["path"][i].tolist() == r["path"], tag
        want_status = d.READ_NO_DECODING if r["loglike"] == "-inf" else d.READ_OK
        assert out["status"][i] == want_status, tag
    return dec


@pytest.mark.parametrize("name", CASES)
def test_gpu_matches_reference_golden(d, name):
    dec = _check_against_golden(d, util.golden_case(name))
    st = dec.stats()
    assert st["fill_launches"] >= 1 and st["traceback_launches"] >= 1


@pytest.mark.parametrize("cluster", [1, 2, 4, 8, 16])
@pytest.mark.parametrize("name", ["l4c4_global_mixed", "l4c4_local_mixed", "mr2l4c4_local", "cfg3_global_indels"])
def test_gpu_every_cluster_size(d, name, cluster):
    """The state partition over the thread-block cluster must not change a single bit."""
    case = util.golden_case(name)
    n_states = util.compiled_for_case(case).t.n_states
    if cluster == 1 and n_states > 4000:
        pytest.skip("does not fit one CTA")
    for tmode in (1, 2):  # duplication columns in shared memory / in global scratch
        if tmode == 1 and cluster <= 2 and n_states > 4000:
            continue
        _check_against_golden(d, case, dict(cluster_size=cluster, t_in_smem_mode=tmode))


# "table" / "s_prev": 1 shared memory, 2 global memory; "partition": 1 index runs, 2 DFS runs, 3 DFS chunks dealt,
# 4 DFS runs sorted; 0 = automatic
@pytest.mark.parametrize("cluster,table,s_prev,partition", [(3, 0, 2, 0), (6, 0, 2, 4), (8, 2, 2, 3), (2, 1, 2, 2), (1, 0, 2, 0),
                                                           (5, 2, 1, 4), (4, 2, 2, 1), (12, 1, 1, 3), (16, 1, 1, 4)])
@pytest.mark.parametrize("name", ["l4c4_local_mixed", "cfg3_global_indels", "cfg4_global_dels"])
def test_gpu_push_placements_and_partitions(d, name, cluster, table, s_prev, partition):
    """S(pos-1) in shared memory / global scratch, transition table in shared / global memory, odd cluster sizes and
    every partition policy of the push kernel, set through the named options: none of it may change a bit."""
    case = util.golden_case(name)
    if cluster == 1 and util.compiled_for_case(case).t.n_states > 4000:
        pytest.skip("does not fit one CTA")
    opts = dict(table=table, s_prev=s_prev, partition=partition)
    try:
        _check_against_golden(d, case, dict(cluster_size=cluster), {k: v for k, v in opts.items() if v})
    except d.DnabError as e:
        if "does not fit" in str(e):
            pytest.skip("requested placement does not fit this machine")
        raise


def test_gpu_retired_pull_kernel_is_refused(d):
    """kernel=3 selected the pull-closure fill kernel, which was retired: the option is refused with an error that
    says so, and the handle keeps decoding with what it had."""
    case = util.golden_case("l4c4_global_mixed")
    dec = d.Decoder(util.compiled_for_case(case), device=0)
    dec.set_option("kernel", 2)
    with pytest.raises(d.DnabError, match="retired"):
        dec.set_option("kernel", 3)
    _check_reads(d, dec, case, "after kernel=3")


@pytest.mark.parametrize("workload,n", [("cfg2", 99), ("cfg5", 300), ("cfg3", 300)])
def test_gpu_fill_kernels_agree_at_batch_scale(d, workload, n):
    """Two independent implementations of the fill (read-batched and one-read-per-cluster push kernel, different
    table formats, different partitions) must agree bit for bit -- log-likelihood, decoded string, traceback
    path -- on a batch far larger than the oracle can check in a test (several waves of clusters or teams, ragged
    lengths, dynamic read scheduling)."""
    import bench
    w = bench.WORKLOADS[workload]
    compiled = util.machine_from_recipe(w["recipe"]).compile(d.ErrorFlags(length=w["length"], global_=True))
    reads = bench.make_reads(w, n, seed=4242)
    outs = []
    for kern in (1, 2):
        dec = d.Decoder(compiled, device=0)
        dec.set_option("kernel", kern)
        outs.append(dec.viterbi(reads, want_path=True))
    a, b = outs
    assert (a["status"] == 0).all() and (b["status"] == 0).all()
    assert a["loglike"].tobytes() == b["loglike"].tobytes()
    assert a["decoded"] == b["decoded"]
    assert all(x.tolist() == y.tolist() for x, y in zip(a["path"], b["path"]))
    # and the decoder does its job: most of these lightly mutated reads decode to a framed bit string
    assert sum(s.startswith("^") and s.endswith("$") for s in a["decoded"]) > 0.9 * n


@pytest.mark.parametrize("opts", [dict(thin_n=0), dict(thin_n=48), dict(t_recompute=0),
                                  dict(queue_cap=40), dict(queue_cap=40, thin_n=100000)])
@pytest.mark.parametrize("name", ["l4c4_global_mixed", "l4c4_local_mixed", "cfg3_global_indels", "cfg4_global_dels",
                                  "cfg2_global_subs"])
def test_gpu_push_kernel_tuning_knobs_same_bits(d, name, opts):
    """How a level's work list is made (bitmap scan, or appended by the previous level's pushers below a size
    threshold -- including a threshold so large that the small append queues overflow), stored (not re-derived)
    duplication cells and a scan queue far smaller than the frontier are schedule / placement choices of the
    push kernel: no bit may change."""
    _check_against_golden(d, util.golden_case(name), options=dict(kernel=2, **opts))


@pytest.mark.parametrize("threads", [32, 96, 256, 1024])
def test_gpu_every_block_size(d, threads):
    _check_against_golden(d, util.golden_case("l4c4_global_mixed"), dict(threads_per_cta=threads))


@pytest.mark.parametrize("tag", ["l4c4_global", "l4c4_local"])
def test_gpu_cells_bit_exact(d, tag):
    z = np.load(f"{util.GOLDEN}/cells_{tag}.npz")
    flags = json.loads(str(z["flags"]))
    compiled = util.compiled_for([str(x) for x in z["recipe"]], flags, bool(z["global_"]))
    dec = d.Decoder(compiled, device=0)
    ll, cells = dec.viterbi_cells(str(z["seq"]))
    assert cells.tobytes() == z["cells"].reshape(cells.shape).tobytes()
    assert util.hexf(ll) == util.hexf(str(z["loglike_hex"]))


def test_gpu_vs_oracle_seeded_batch(d):
    """A few hundred seeded mutated reads on l4c4 (global and local): GPU == oracle, bit for bit."""
    from benchdata import synth
    rng = np.random.default_rng(20261018)
    pool = [r["seq"] for r in util.golden_case("l4c4_global_mixed")["reads"]]
    reads = [synth.mutate(pool[i % len(pool)], rng, sub_rate=0.03, dup_rate=0.01, max_dup=2, del_rate=0.01, max_del=4)
             for i in range(192)]
    reads += ["", "A", "ACGT" * 3]  # empty and very short reads ride along in the same batch
    for global_ in (True, False):
        compiled = util.compiled_for(["l4c4"], dict(length=4), global_)
        dec = d.Decoder(compiled, device=0)
        out = dec.viterbi(reads, want_path=True)
        for i, s in enumerate(reads):
            o = util.oracle_viterbi(compiled, s)
            assert out["decoded"][i] == o["decoded"], (global_, i)
            assert util.hexf(out["loglike"][i]) == util.hexf(o["loglike"]), (global_, i)
            assert out["path"][i].tolist() == o["path"], (global_, i)


def test_gpu_ragged_batch_order_and_chunking(d):
    """Results come back in input order whatever the batch composition; decoding a read alone or
    inside a ragged batch gives the same bits."""
    case = util.golden_case("l4c4_global_mixed")
    compiled = util.compiled_for_case(case)
    dec = d.Decoder(compiled, device=0)
    reads = [r["seq"] for r in case["reads"]]
    ragged = [reads[0][:5], reads[1], "", reads[2][:77], reads[3]] * 7
    whole = dec.viterbi(ragged)
    for i, s in enumerate(ragged):
        one = dec.viterbi([s])
        assert one["decoded"][0] == whole["decoded"][i]
        assert util.hexf(one["loglike"][0]) == util.hexf(whole["loglike"][i])


def test_gpu_decode_fasta_drop_in(d, tmp_path):
    """decodeFastSeqs drop-in: multi-line records, lower case, names kept, input order."""
    case = util.golden_case("kat186")  # the reference's 3-line record with a deleted base
    seq = case["reads"][0]["seq"]
    fa = tmp_path / "reads.fa"
    fa.write_text(">first some comment\n" + seq[:30] + "\n" + seq[30:60].lower() + "\n" + seq[60:] + "\n>second\n" + seq + "\n")
    dec = d.Decoder(util.compiled_for_case(case), device=0)
    got = dec.decode_fasta(fa)
    assert [g[0] for g in got] == ["first", "second"]
    assert got[0][1] == got[1][1] == case["reads"][0]["decoded"]
    assert util.hexf(got[0][2]) == util.hexf(case["reads"][0]["loglike_hex"])


def test_gpu_cli_matches_reference_cli_output(d, tmp_path):
    """bin/dnastore-b200 -V prints what the reference prints for its own known-answer test."""
    import os
    import subprocess
    case = util.golden_case("kat147")
    fa = tmp_path / "hello.fa"
    fa.write_text(">hello\n" + case["reads"][0]["seq"] + "\n")
    exe = os.path.join(util.ROOT, "bin", "dnastore-b200")
    out = subprocess.run([exe, "-v0", "--load-machine", util.machine_path("l4c4"), "--decode-viterbi", str(fa),
                          "--error-sub-prob", "0", "--error-dup-prob", "0", "--error-del-open", "0", "--error-global",
                          "--raw"], capture_output=True, text=True, check=True).stdout
    assert out == case["reads"][0]["decoded"] + "\n"


# ----------------------------------------------------------------------------------------------
# round 2: the read-batched kernel (viterbi_fill_batch.cu, option kernel=1) and the benchmark-scale goldens
# ----------------------------------------------------------------------------------------------
R2_CASES = [c["name"] for c in util.load_golden_r2()["cases"]]


def _check_reads(d, dec, case, tag):
    reads = [r["seq"] for r in case["reads"]]
    out = dec.viterbi(reads, want_path=True)
    for i, r in enumerate(case["reads"]):
        assert out["decoded"][i] == r["decoded"], (tag, r["name"])
        assert util.hexf(out["loglike"][i]) == util.hexf(r["loglike_hex"]), (tag, r["name"])
        assert out["path"][i].tolist() == r["path"], (tag, r["name"])
        assert out["status"][i] == (d.READ_NO_DECODING if r["loglike"] == "-inf" else d.READ_OK), (tag, r["name"])


@pytest.mark.parametrize("name", R2_CASES)
def test_gpu_round2_goldens_default_kernel(d, name):
    """The benchmark read distributions at full length -- 64 reads of the headline 46,670-state workload, 32 of each
    other BASELINE machine, 8 of dnastore-l10 -- against the UNMODIFIED reference: log-likelihood bits, decoded string,
    traceback path, through whichever kernel the decoder picks by itself."""
    case = util.golden_r2_case(name)
    _check_reads(d, d.Decoder(util.compiled_for_case(case), device=0), case, name)


@pytest.mark.parametrize("async_closure", [0, 1])
@pytest.mark.parametrize("name", CASES + R2_CASES)
def test_gpu_batch_kernel_matches_reference_golden(d, name, async_closure):
    """Every golden case through the read-batched kernel (32 reads are the lanes of a warp; teams of 1-148 CTAs), with
    the closure in breadth-first levels and without level barriers."""
    case = util.golden_case(name) if name in CASES else util.golden_r2_case(name)
    dec = d.Decoder(util.compiled_for_case(case), device=0)
    dec.set_option("kernel", 1)
    dec.set_option("async_closure", async_closure)
    try:
        info = dec.batch_info()
    except d.DnabError as e:
        pytest.skip(f"machine does not fit the shared memory of the GPU at 32 reads per group: {e}")
    assert info["enabled"] == 1 and info["reads_per_group"] == 32
    _check_reads(d, dec, case, (name, info["team_size"]))


@pytest.mark.parametrize("async_closure", [0, 1])
@pytest.mark.parametrize("team,warps", [(1, 16), (1, 32), (2, 24), (3, 16), (7, 32), (16, 24)])
@pytest.mark.parametrize("name", ["l4c4_global_mixed", "l4c4_local_mixed", "l4c4_len12_local", "mr2l4c4_local"])
def test_gpu_batch_kernel_every_team_size(d, name, team, warps, async_closure):
    """How many CTAs share a group (and how their states are partitioned), how many warps a CTA has, and whether the
    closure runs in breadth-first levels or without level barriers are placement / schedule choices: no bit may change."""
    case = util.golden_case(name)
    dec = d.Decoder(util.compiled_for_case(case), device=0)
    dec.set_option("kernel", 1)
    dec.set_option("team_size", team)
    dec.set_option("warps_per_cta", warps)
    dec.set_option("async_closure", async_closure)
    try:
        info = dec.batch_info()
    except d.DnabError:
        pytest.skip("this team size cannot hold the machine")
    assert info["team_size"] == team
    _check_reads(d, dec, case, (name, team, warps))


@pytest.mark.parametrize("classes", [1, 5, 32])
@pytest.mark.parametrize("name", ["mr2l4c4_local", "cfg4_global_dels", "cfg5_l8_local", "cfg2_global_subs"])
def test_gpu_batch_kernel_notification_classes_same_bits(d, name, classes):
    """Teams: a notified CTA re-relaxes the transitions from other CTAs of the notified classes of its states only (32
    classes by default; 1 = every such transition): a schedule choice, no bit may change."""
    case = util.golden_case(name)
    dec = d.Decoder(util.compiled_for_case(case), device=0)
    dec.set_option("kernel", 1)
    dec.set_option("notify_classes", classes)
    _check_reads(d, dec, case, name)


@pytest.mark.parametrize("kernel", [0, 1])
def test_gpu_cfg2_cells_hash(d, kernel):
    """Every DP cell of a short read on the 46,670-state machine (global and local mode) hashes to the reference's
    matrix: cell-exactness on a 4-CTA cluster (push kernel) and on a 148-CTA team (read-batched kernel)."""
    import hashlib
    for c in util.load_golden_r2()["cells"]:
        dec = d.Decoder(util.compiled_for(c["recipe"], c["flags"], c["global_"]), device=0)
        dec.set_option("kernel", kernel)
        ll, cells = dec.viterbi_cells(c["seq"])
        assert cells.size == c["n_cells"]
        assert hashlib.sha256(cells.tobytes()).hexdigest() == c["sha256"], (c["name"], kernel)
        assert util.hexf(ll) == util.hexf(c["loglike_hex"])


@pytest.mark.parametrize("kernel", [1, 2])
def test_gpu_production_kernel_end_cells_by_prefix(d, kernel):
    """The cell dump runs an instrumented instantiation; the PRODUCTION instantiation is held to the reference's cells
    through a debug-free path: the log-likelihood of the p-base prefix of a read is the cell S(end, p) of the full
    read's matrix (global mode), so decoding every prefix in one batch checks one cell per column, bit for bit."""
    z = np.load(f"{util.GOLDEN}/cells_l4c4_global.npz")
    flags = json.loads(str(z["flags"]))
    compiled = util.compiled_for([str(x) for x in z["recipe"]], flags, True)
    seq = str(z["seq"])
    n, k = compiled.t.n_states, compiled.t.k
    cells = z["cells"].reshape(len(seq) + 1, n, k + 2)
    dec = d.Decoder(compiled, device=0)
    dec.set_option("kernel", kernel)
    out = dec.viterbi([seq[:p] for p in range(len(seq) + 1)])
    for p in range(len(seq) + 1):
        assert util.hexf(out["loglike"][p]) == util.hexf(float(cells[p, n - 1, 0])), p


@pytest.mark.parametrize("workload,n", [("cfg1", 3000), ("cfg4", 400), ("cfg2", 99), ("cfg5", 300)])
def test_gpu_batch_and_push_kernels_agree_at_batch_scale(d, workload, n):
    """Read-batched kernel (groups of 32 reads sorted by length, several groups per team, ragged last group) against
    the one-read-per-cluster push kernel on a batch far larger than the goldens: same bits, same strings, same paths."""
    import bench
    w = bench.WORKLOADS[workload]
    compiled = util.machine_from_recipe(w["recipe"]).compile(d.ErrorFlags(length=w["length"], global_=True))
    reads = bench.make_reads(w, n, seed=777)
    reads[3] = reads[3][:17]  # ragged: short, empty and long reads share groups
    reads[5] = ""
    outs = []
    for kern in (1, 2):
        dec = d.Decoder(compiled, device=0)
        dec.set_option("kernel", kern)
        outs.append(dec.viterbi(reads, want_path=True))
    a, b = outs
    assert a["loglike"].tobytes() == b["loglike"].tobytes()
    assert a["decoded"] == b["decoded"]
    assert (a["status"] == b["status"]).all()
    assert all(x.tolist() == y.tolist() for x, y in zip(a["path"], b["path"]))


# ----------------------------------------------------------------------------------------------
# several devices and the ingest pipeline (dnab_multi_decoder, dnab_decode_fasta[_multi])
# ----------------------------------------------------------------------------------------------
def _two_devices():
    import torch
    return [0, 1] if torch.cuda.device_count() >= 2 else [0, 0]  # the same GPU twice still runs two decoders and two host threads


def test_gpu_multi_decoder_matches_goldens(d):
    """The product's multi-GPU entry (dnab_viterbi_batch_multi: chunks handed to one host thread and decoder per
    device, results in input order) against the reference goldens, with two devices when the box has them."""
    for name in ("cfg1_bench", "cfg4_bench", "cfg2_bench"):
        case = util.golden_r2_case(name)
        md = d.MultiDecoder(util.compiled_for_case(case), _two_devices())
        md.set_option("chunk_reads", 8)  # many small chunks: both decoders get work, order must survive
        reads = [r["seq"] for r in case["reads"]]
        out = md.viterbi(reads)
        assert md.stats()["chunks"] == (len(reads) + 7) // 8
        for i, r in enumerate(case["reads"]):
            assert out["decoded"][i] == r["decoded"], (name, i)
            assert util.hexf(out["loglike"][i]) == util.hexf(r["loglike_hex"]), (name, i)


def test_gpu_fasta_pipeline_chunks_gzip_fastq_and_overflow(d, tmp_path):
    """dnab_decode_fasta_multi: the file is parsed in bounded chunks by a producer thread while earlier chunks are
    decoded; gzip + FASTQ + multi-line records; a decoded-string slot far too small on the first attempt makes every
    read overflow and be decoded again with a larger slot (only those reads).  Names, order and bits as the reference."""
    import gzip
    case = util.golden_r2_case("cfg1_bench")
    fq = tmp_path / "reads.fq.gz"
    with gzip.open(fq, "wt") as f:
        for r in case["reads"]:
            s = r["seq"]
            f.write(f"@{r['name']} comment\n{s[:50]}\n{s[50:].lower()}\n+\n{'I' * len(s)}\n")
    md = d.MultiDecoder(util.compiled_for_case(case), _two_devices())
    md.set_option("chunk_reads", 5)
    md.set_option("decoded_slot_bytes", 16)
    got = md.decode_fasta(fq)
    st = md.stats()
    assert st["reads"] == len(case["reads"]) and st["chunks"] == (len(case["reads"]) + 4) // 5
    assert st["overflow_reruns"] >= len(case["reads"])
    assert [g[0] for g in got] == [r["name"] for r in case["reads"]]
    for g, r in zip(got, case["reads"]):
        assert g[1] == r["decoded"] and util.hexf(g[2]) == util.hexf(r["loglike_hex"]) and g[3] == d.READ_OK
    # one device, default chunking, through dnab_decode_fasta
    got1 = d.Decoder(util.compiled_for_case(case), device=0).decode_fasta(fq)
    assert got1 == got


def test_gpu_fasta_pipeline_reports_bad_base(d, tmp_path):
    """A non-ACGT character terminates the reference (src/fastseq.cpp:25-39); here it is an error from the producer
    thread that names the record."""
    fa = tmp_path / "bad.fa"
    fa.write_text(">ok\nACGT\n>broken\nACGNT\n")
    dec = d.Decoder(util.compiled_for(["l4c4"], dict(length=4), True), device=0)
    with pytest.raises(d.DnabError, match="Unknown symbol N in sequence broken"):
        dec.decode_fasta(fa)


def test_gpu_cli_devices_flag(d, tmp_path):
    import os
    import subprocess
    case = util.golden_r2_case("cfg1_bench")
    fa = tmp_path / "r.fa"
    fa.write_text("".join(f">{r['name']}\n{r['seq']}\n" for r in case["reads"]))
    exe = os.path.join(util.ROOT, "bin", "dnastore-b200")
    devs = ",".join(str(x) for x in _two_devices())
    out = subprocess.run([exe, "-v0", "-l", "4", "--load-machine", util.machine_path("l4c4"), "--decode-viterbi", str(fa),
                          "--error-global", "--raw", "--devices", devs], capture_output=True, text=True, check=True).stdout
    assert out.split("\n")[:-1] == [r["decoded"] for r in case["reads"]]


def test_gpu_rejects_malformed_batches(d):
    """Caller arrays are validated on the host before any launch (a misaligned offset would fault the context)."""
    dec = d.Decoder(util.compiled_for(["l4c4"], dict(length=4), True), device=0)
    packed, off, ln = d.pack_reads(["ACGTACGT", "TTTT"])
    bad = off.copy()
    bad[1] += 4
    with pytest.raises(d.DnabError):
        dec.viterbi_packed(packed, bad, ln)
    neg = ln.copy()
    neg[0] = -3
    with pytest.raises(d.DnabError):
        dec.viterbi_packed(packed, off, neg)
    assert dec.viterbi(["ACGTACGT"])["status"][0] == d.READ_OK  # the handle is still usable
