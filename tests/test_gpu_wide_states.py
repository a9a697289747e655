"""Machines with wide states: more incoming candidates than a 1-byte predecessor record can name, or more than 255
successors (dnastore_b200/csrc/viterbi_device.cuh).  Their S and D records keep a second byte in a side plane; every
front end decodes them bit-exact with the oracle, which has no degree limit.

The machines are generated here, seeded: (a) a hub with 300 null in-transitions, (b) a join with 160 emitting
in-transitions (320 D candidates), (c) a state with 300 successors whose branches rejoin through 300 emitting
transitions, (d) an outer machine with a 1200-way selector composed onto l4c4 (real k-mer contexts and T cells)."""
import gzip
import json
import os
import subprocess

import numpy as np
import pytest

import dnab_testutil as util

BASES = "ACGT"
FLAGS = dict(length=4, sub=.01, iv=10., dup=.001, delopen=.001, delext=.01)  # = the CLI's defaults with -l 4


class _Builder:
    def __init__(self):
        self.trans = []

    def state(self):
        self.trans.append([])
        return len(self.trans) - 1

    def add(self, src, dst, inp=None, out=None):
        t = {"to": dst}
        if inp is not None:
            t["in"] = inp
        if out is not None:
            t["out"] = out
        self.trans[src].append(t)

    def json(self):
        return json.dumps({"state": [{"n": i, "id": f"s{i}", "trans": t} for i, t in enumerate(self.trans)]})


def _code(i, n):
    return "".join(BASES[(i >> (2 * j)) & 3] for j in range(n))


def _fan(n, code_len, join_emits, trie=False):
    """State 0 -> n branches (each a chain emitting a distinct code, its first state a distinct successor of state 0;
    or, with `trie`, the codes share their prefixes) -> one join state (through n null transitions, or n emitting ones:
    the last base of every code) -> a short tail."""
    b = _Builder()
    s0 = b.state()
    ends = []
    node = {}
    for i in range(n):
        prev = s0
        chain = code_len - 1 if join_emits else code_len
        for j in range(chain):
            key = _code(i, code_len)[:j + 1]
            if trie and key in node:
                prev = node[key]
                continue
            nxt = b.state()
            b.add(prev, nxt, inp="01"[(i >> j) & 1], out=_code(i, code_len)[j])
            node[key] = prev = nxt
        ends.append((prev, _code(i, code_len)[-1]))
    join = b.state()
    for prev, last in ends:
        b.add(prev, join, out=last if join_emits else None)
    prev = join
    for ch in "TTT":
        nxt = b.state()
        b.add(prev, nxt, out=ch)
        prev = nxt
    return b.json()


def _selector(n=1200, bits=11, suffix="01" * 12):
    """Outer machine for l4c4: '^', then one of n 11-bit codes (the selector state has n successors), a common suffix,
    a null join of the n branches, '$'.  After composition the join is spread over the inner states that the branches
    end in; with 1200 branches the largest of them still has more than 254 candidates."""
    b = _Builder()
    s0 = b.state()
    sel = b.state()
    b.add(s0, sel, inp="^", out="^")
    ends = []
    for i in range(n):
        prev = sel
        for ch in format(i, f"0{bits}b") + suffix:
            nxt = b.state()
            b.add(prev, nxt, inp=ch, out=ch)
            prev = nxt
        ends.append(prev)
    join = b.state()
    for e in ends:
        b.add(e, join)
    end = b.state()
    b.add(join, end, inp="$", out="$")
    return b.json()


MACHINES = ("a_null_hub", "b_emit_join", "c_fan_out", "d_selector_l4c4")


def _machine(name):
    import dnastore_b200 as d
    if name == "a_null_hub":
        return d.Machine.from_json(_fan(300, 5, False))
    if name == "b_emit_join":
        return d.Machine.from_json(_fan(160, 5, True, trie=True))  # (small enough for one CTA; 4 bases tell branches apart)
    if name == "c_fan_out":
        return d.Machine.from_json(_fan(300, 5, True))
    return d.Machine.compose(d.Machine.from_json(_selector()), d.Machine.from_file(util.machine_path("l4c4")))


_COMPILED = {}


def _compiled(name, global_=True):
    key = (name, global_)
    if key not in _COMPILED:
        # (b): deletions cheaper than substitutions, so that a deleted join base is explained through the join's D cell
        flags = dict(FLAGS, sub=.001, delopen=.05) if name == "b_emit_join" else FLAGS
        _COMPILED[key] = _machine(name).compile(util.error_flags(flags, global_))
    return _COMPILED[key]


def _degrees(a):
    n = a["n_states"]
    n_e = np.diff(a["emit_off"]).astype(np.int64)
    n_n = np.diff(a["null_off"]).astype(np.int64)
    n_out = np.bincount(np.concatenate([a["emit_src"], a["null_src"]]).astype(np.int64), minlength=n)
    succ = np.zeros(n, dtype=np.int64)
    pairs = set()
    for dst in range(n):
        for s in a["emit_src"][a["emit_off"][dst]:a["emit_off"][dst + 1]]:
            pairs.add((int(s), dst))
        for s in a["null_src"][a["null_off"][dst]:a["null_off"][dst + 1]]:
            pairs.add((int(s), dst))
    for s, _ in pairs:
        succ[s] += 1
    return n_e, n_n, n_out, succ


def _wide(n_e, n_n, n_out):
    """The wide-state rule of viterbi_device.cuh (stateIsWide)."""
    return (n_e > 126) | (n_e + n_n + 2 > 254) | (2 * n_e + n_n > 254) | (n_out > 255)


def _walk(a, rng):
    """A random path from state 0 to the end state through the compiled tables: the bases it emits, and for every base
    the state its transition enters."""
    n = a["n_states"]
    outs = [[] for _ in range(n)]
    for dst in range(n):
        for e in range(a["emit_off"][dst], a["emit_off"][dst + 1]):
            outs[a["emit_src"][e]].append((dst, int(a["emit_base"][e])))
        for e in range(a["null_off"][dst], a["null_off"][dst + 1]):
            outs[a["null_src"][e]].append((dst, None))
    for _ in range(1000):
        s, seq, into = 0, [], []
        while s != n - 1 and outs[s] and len(seq) < 400:
            dst, base = outs[s][rng.integers(len(outs[s]))]
            if base is not None:
                seq.append(BASES[base])
                into.append(dst)
            s = dst
        if s == n - 1:
            return "".join(seq), into
    raise AssertionError("no path to the end state")


_READS = {}


def _reads(name, count=48, seed=20261021):
    """Seeded reads of the machine: random paths, lightly mutated; every other read loses the base that enters the
    state with the most emitting in-transitions (so that its D record is used there)."""
    if name not in _READS:
        from benchdata import synth
        a = _compiled(name).arrays()
        n_e = np.diff(a["emit_off"])
        join = int(np.argmax(n_e))
        rng = np.random.default_rng(seed + MACHINES.index(name))
        reads = []
        for i in range(count):
            seq, into = _walk(a, rng)
            if i % 2 and join in into:
                p = into.index(join)
                seq = seq[:p] + seq[p + 1:]
            else:
                seq = synth.mutate(seq, rng, sub_rate=0.02, dup_rate=0.005, max_dup=2, del_rate=0.005, max_del=2).upper()
            reads.append(seq)
        _READS[name] = reads
    return _READS[name]


def _record_indices(a, path):
    """Candidate index chosen by every S and D traceback step of an oracle path (reference order,
    src/viterbi.cpp:251-276): S = [emit..., null..., delEnd, T->S, local start], D = [2 per emit edge, null...]."""
    got = []
    for (s, pos, mut), (s2, pos2, mut2) in zip(path, path[1:]):
        if mut >= 2:
            continue
        e0, e1 = int(a["emit_off"][s]), int(a["emit_off"][s + 1])
        n0, n1 = int(a["null_off"][s]), int(a["null_off"][s + 1])
        n_e, n_in = e1 - e0, (e1 - e0) + (n1 - n0)
        emit = [int(x) for x in a["emit_src"][e0:e1]]
        null = [int(x) for x in a["null_src"][n0:n1]]
        if mut == 0:
            if s2 == s and mut2 == 1:
                got.append(n_in)
            elif s2 == s and mut2 == 2:
                got.append(n_in + 1)
            elif pos2 == pos - 1 and mut2 == 0:
                got.append(emit.index(s2))
            else:
                got.append(n_e + null.index(s2))
        else:
            if pos2 == pos and s2 in emit and mut2 in (0, 1) and (mut2 == 0 or s2 not in null):
                got.append(2 * emit.index(s2) + (1 if mut2 == 0 else 0))
            else:
                got.append(2 * n_e + null.index(s2))
    return got


# ----------------------------------------------------------------------------------------------
# CPU: the generator and the reads
# ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", MACHINES)
def test_wide_machine_generator(name):
    """The degrees each machine promises; no null cycle (compilation succeeds); wide states present; and the seeded reads
    really take the second record byte: some oracle traceback step chooses a candidate >= 255, some one below."""
    c = _compiled(name)
    a = c.arrays()
    n_e, n_n, n_out, succ = _degrees(a)
    if name == "a_null_hub":
        assert n_n.max() >= 300
    if name == "b_emit_join":
        assert n_e.max() >= 130 and (2 * n_e + n_n).max() > 254
    if name == "c_fan_out":
        assert succ.max() >= 300 and n_e.max() >= 300
    if name == "d_selector_l4c4":
        assert succ.max() >= 256 and (n_e + n_n + 3).max() > 254 and a["k"] > 0 and a["mdl"].max() > 0
    assert _wide(n_e, n_n, n_out).sum() > 0
    chosen = []
    for seq in _reads(name):
        o = util.oracle_viterbi(c, seq)
        assert o["rc"] == 0 and o["loglike"] > -np.inf
        chosen += _record_indices(a, o["path"])
    assert max(chosen) >= 255 and min(chosen) < 255


# ----------------------------------------------------------------------------------------------
# GPU
# ----------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def d():
    import dnastore_b200
    import torch
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return dnastore_b200


KERNELS = {
    "auto": {},
    "batched": dict(kernel=1),
    "batched_team1": dict(kernel=1, team_size=1),
    "batched_team6": dict(kernel=1, team_size=6),
    "push": dict(kernel=2),
    "push_cluster2": dict(kernel=2, cluster_size=2),
}
# placements a machine fits: only (b) fits one CTA; (d) (45,316 states) needs a team of most of the GPU, and four CTAs
# per read in the push kernel, which it picks itself
PLACEMENTS = [(name, kernel) for name in MACHINES for kernel in KERNELS
              if (kernel != "batched_team1" or name == "b_emit_join")
              and (name != "d_selector_l4c4" or kernel not in ("batched_team6", "push_cluster2"))]

_ORACLE = {}


def _oracle(name, global_, i):
    key = (name, global_, i)
    if key not in _ORACLE:
        _ORACLE[key] = util.oracle_viterbi(_compiled(name, global_), _reads(name)[i])
    return _ORACLE[key]


@pytest.mark.gpu
@pytest.mark.parametrize("global_", [True, False], ids=["global", "local"])
@pytest.mark.parametrize("name,kernel", PLACEMENTS)
def test_gpu_wide_parity_with_oracle(d, name, global_, kernel):
    """Loglike bit-equal, decoded string and path equal to the oracle on every kernel and in both modes."""
    c = _compiled(name, global_)
    reads = _reads(name)
    dec = d.Decoder(c, device=0)
    for key, value in KERNELS[kernel].items():
        dec.set_option(key, value)
    out = dec.viterbi(reads, want_path=True)
    if kernel.startswith("batched"):
        assert dec.batch_info()["wide_states"] > 0
    for i in range(len(reads)):
        o = _oracle(name, global_, i)
        assert util.hexf(out["loglike"][i]) == util.hexf(o["loglike"]), (name, kernel, i)
        assert out["decoded"][i] == o["decoded"], (name, kernel, i)
        assert out["path"][i].tolist() == o["path"], (name, kernel, i)


@pytest.mark.gpu
@pytest.mark.parametrize("kernel", ["auto", "push"])
@pytest.mark.parametrize("name", ["a_null_hub", "d_selector_l4c4"])
def test_gpu_wide_cells_bit_exact(d, name, kernel):
    c = _compiled(name)
    seq = _reads(name)[1]
    dec = d.Decoder(c, device=0)
    for key, value in KERNELS[kernel].items():
        dec.set_option(key, value)
    ll, cells = dec.viterbi_cells(seq)
    o = util.oracle_viterbi(c, seq, want_cells=True)
    assert cells.tobytes() == o["cells"].tobytes()
    assert util.hexf(ll) == util.hexf(o["loglike"])


def _two_devices():
    import torch
    return [0, 1] if torch.cuda.device_count() >= 2 else [0, 0]


@pytest.mark.gpu
def test_gpu_wide_front_ends(d, tmp_path):
    """dnab_viterbi_batch_multi, dnab_decode_fasta on a gzip FASTA and bin/dnastore-b200 -V --raw on machine (d)."""
    name = "d_selector_l4c4"
    c = _compiled(name)
    reads = _reads(name)
    want = [_oracle(name, True, i)["decoded"] for i in range(len(reads))]
    md = d.MultiDecoder(c, _two_devices())
    md.set_option("chunk_reads", 16)
    assert md.viterbi(reads)["decoded"] == want
    fa = tmp_path / "reads.fa.gz"
    with gzip.open(fa, "wt") as f:
        f.write("".join(f">r{i}\n{s}\n" for i, s in enumerate(reads)))
    got = d.Decoder(c, device=0).decode_fasta(fa)
    assert [g[0] for g in got] == [f"r{i}" for i in range(len(reads))]
    assert [g[1] for g in got] == want
    mj = tmp_path / "selector_l4c4.json"
    mj.write_text(_machine(name).to_json())
    exe = os.path.join(util.ROOT, "bin", "dnastore-b200")
    out = subprocess.run([exe, "-v0", "-l", "4", "--load-machine", str(mj), "--decode-viterbi", str(fa), "--error-global",
                          "--raw"], capture_output=True, text=True, check=True).stdout
    assert out.split("\n")[:-1] == want


def _too_many_candidates(n_null=65533):
    """A state with n_null parallel null in-transitions: nE + nN + 3 = 65536 S candidates, one more than a wide record
    can name."""
    b = _Builder()
    s0, s1, s2, s3 = b.state(), b.state(), b.state(), b.state()
    b.add(s0, s1, inp="0", out="A")
    for _ in range(n_null):
        b.add(s1, s2)
    b.add(s2, s3, out="C")
    return b.json()


@pytest.mark.gpu
@pytest.mark.parametrize("kernel", ["auto", "push"])
def test_gpu_wide_refuses_records_past_16_bits(d, kernel):
    import dnastore_b200
    c = dnastore_b200.Machine.from_json(_too_many_candidates()).compile(util.error_flags(FLAGS, True))
    assert int(np.diff(c.arrays()["null_off"]).max()) == 65533
    dec = d.Decoder(c, device=0)
    for key, value in KERNELS[kernel].items():
        dec.set_option(key, value)
    with pytest.raises(d.DnabError, match="predecessor records hold at most 65535 candidates") as e:
        dec.viterbi(["AC"])
    assert e.value.code == -1  # DNAB_EINVAL
    ok = _compiled("a_null_hub")
    seq = _reads("a_null_hub")[0]
    out = d.Decoder(ok, device=0).viterbi([seq])
    assert util.hexf(out["loglike"][0]) == util.hexf(util.oracle_viterbi(ok, seq)["loglike"])
