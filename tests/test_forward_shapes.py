"""The forward-backward kernel (forward_kernels.cu) at the launch shapes, machines and reads where it can go wrong.

Two references:
  * the specification, oracle/forward_oracle.c: the GPU must give the same log-likelihood bits, sweeps and status, and
    counts and posteriors within 1e-9 (the kernel sums the states in another fixed order);
  * an EXACT computation in probability space (exact_fwdback below): float64, a direct solve of every column's
    closure, no table log_sum_exp, no sweep limit.  The log-likelihood, the expected counts and the posteriors all
    come out of one autograd call, so they do not rest on the hand-derived backward recursion the oracle and the kernel
    share.

The launch shapes are forced through the decoder options "fwd_threads" (CTA width) and "fwd_blocks" (grid cap), and
checked through dnab_decoder_stats.last_fwd_threads / last_fwd_blocks, so that an option that is ignored cannot make a
test pass that tests nothing.
"""
import os
from concurrent.futures import ThreadPoolExecutor

import ctypes as C
import numpy as np
import pytest
import torch

import dnab_testutil as util
import test_gpu_wide_states as wide
from test_forward import exact_forward

FLAGS = dict(length=4, sub=.01, iv=10., dup=.001, delopen=.001, delext=.01)  # the CLI's defaults with -l 4

# Exact reference against the specification, largest differences over the 22 reads of
# test_exact_reference_against_specification (l4c4 global and local, mr2l4c4, a k = 0 machine, the 6-symbol machine;
# 0 to 110 bases, many indels):
#   log-likelihood  exact - oracle up to 7.7e-4 (the table log_sum_exp drops terms below e^-10; never above exact)
#   counts          |oracle - exact| up to 5.3e-4 * max(1, |exact|)   (3.0e-2 absolute, on an nSub near 60)
#   posteriors      |oracle - exact| up to 7.0e-4
# The bounds are 2.6, 3.8 and 4.3 times these:
LL_TOL = 2e-3
COUNT_TOL = 2e-3   # relative to max(1, |exact count|)
POST_TOL = 3e-3


# ----------------------------------------------------------------------------------------------
# the exact reference
# ----------------------------------------------------------------------------------------------
def exact_fwdback(compiled, seq, classes):
    """Probability-space forward pass in float64 with the error-model log-scores and per-base class weights as autograd
    leaves.  Returns (loglike, counts[5 + k + 16], post[L, n_classes]):
      * counts = d loglike / d (delOpen, tanDup, noGap, delExtend, delEnd, len[k], sub[16]): the expected number of
        uses of each event, in the order of dnab_fwdback_counts_batch;
      * post[p, c] = d loglike / d theta[p, c], where every move that consumes read base p is weighted by
        exp(theta[p, c]) (theta = 0) with c the class of the move: the input symbol of an emitting transition, or "+"
        for both duplication moves (T0 -> S, T(i+1) -> T(i)).
    The within-column closure [S; D] = A^-1 [s0; 0], A = [[I - Nn, -pEnd I], [-pOpen E, I - pExt E - Nn]] (the matrix
    of test_forward.exact_forward), is factored once with lu_factor; lu_solve gives the S rows of A^-1 restricted to
    the S right-hand side, and every column is then a product with that block.  Columns are rescaled by their maximum
    (a detached constant), so nothing underflows and the gradients are unchanged."""
    a = compiled.arrays()
    N, k, L = a["n_states"], a["k"], len(seq)
    f64 = torch.float64
    eo, no = a["emit_off"].astype(np.int64), a["null_off"].astype(np.int64)
    ed = torch.from_numpy(np.repeat(np.arange(N), np.diff(eo)))
    nd = torch.from_numpy(np.repeat(np.arange(N), np.diff(no)))
    es = torch.from_numpy(a["emit_src"].astype(np.int64))
    ns = torch.from_numpy(a["null_src"].astype(np.int64))
    ew = torch.from_numpy(np.exp(a["emit_score"]))
    nw = torch.from_numpy(np.exp(a["null_score"]))
    eb = torch.from_numpy(a["emit_base"].astype(np.int64))
    ctx = torch.from_numpy(a["ctx"].astype(np.int64).reshape(N, k))
    has = [torch.from_numpy(a["mdl"].astype(np.int64) > i) for i in range(k)]
    ecls = torch.tensor([classes.index(chr(c)) if c else 0 for c in a["emit_in"]], dtype=torch.int64)
    dup = len(classes) - 1
    leaves = torch.tensor([a["delOpen"], a["tanDup"], a["noGap"], a["delExtend"], a["delEnd"], *a["len"], *a["sub"]],
                          dtype=f64, requires_grad=True)
    theta = torch.zeros((L, len(classes)), dtype=f64, requires_grad=True)
    pOpen, pDup, pNoGap, pExt, pEnd = (leaves[i].exp() for i in range(5))
    pLen = leaves[5:5 + k].exp()
    sub = leaves[5 + k:].exp().reshape(4, 4)
    E = torch.zeros((N, N), dtype=f64).index_put_((ed, es), ew, accumulate=True)
    Nn = torch.zeros((N, N), dtype=f64).index_put_((nd, ns), nw, accumulate=True)
    eye = torch.eye(N, dtype=f64)
    A = torch.cat([torch.cat([eye - Nn, -pEnd * eye], 1), torch.cat([-pOpen * E, eye - pExt * E - Nn], 1)], 0)
    LU, piv = torch.linalg.lu_factor(A)
    closure = torch.linalg.lu_solve(LU, piv, torch.cat([eye, torch.zeros((N, N), dtype=f64)], 0))[:N]  # S <- s0
    tok = torch.from_numpy(util.tokens(seq).astype(np.int64))
    zero = torch.zeros(N, dtype=f64)
    s = torch.ones(N, dtype=f64) if a["local"] else torch.nn.functional.one_hot(torch.tensor(0), N).to(f64)
    T = [zero] * k
    logscale = torch.zeros((), dtype=f64)
    for pos in range(L + 1):
        if pos == 0:
            s = closure @ s
        else:
            x, w = tok[pos - 1], theta[pos - 1].exp()
            s0 = torch.zeros(N, dtype=f64).index_add(0, ed, s[es] * ew * pNoGap * sub[eb, x] * w[ecls])
            if k:
                s0 = s0 + torch.where(has[0], T[0] * sub[ctx[:, 0], x], zero) * w[dup]
            shifted = [torch.where(has[i + 1], T[i + 1] * sub[ctx[:, i + 1], x], zero) * w[dup] for i in range(k - 1)] + [zero]
            s = closure @ s0
            T = [shifted[i] + torch.where(has[i], s * pDup * pLen[i], zero) for i in range(k)]
        scale = s.detach().max()
        if scale > 0:
            s, T, logscale = s / scale, [t / scale for t in T], logscale + scale.log()
    total = s.sum() if a["local"] else s[N - 1]
    ll = total.log() + logscale
    g_leaves, g_theta = torch.autograd.grad(ll, [leaves, theta], allow_unused=True)
    post = g_theta.numpy() if g_theta is not None else np.zeros((L, len(classes)))
    return float(ll.detach()), g_leaves.numpy(), post


def assert_near_exact(exact, loglike, counts, post, what):
    """The specification (or the GPU, which equals it to 1e-9) against the exact reference, within the calibrated
    bounds at the top of the file."""
    ll_x, counts_x, post_x = exact
    assert loglike <= ll_x + 1e-9 * max(1.0, abs(ll_x)), (what, loglike, ll_x)
    assert ll_x - loglike < LL_TOL, (what, loglike, ll_x)
    if counts is not None:
        bad = np.abs(counts - counts_x) > COUNT_TOL * np.maximum(1.0, np.abs(counts_x))
        assert not bad.any(), (what, np.flatnonzero(bad), counts[bad], counts_x[bad])
    if post is not None:
        assert post.shape == post_x.shape, (what, post.shape, post_x.shape)
        assert len(post) == 0 or np.abs(post - post_x).max() < POST_TOL, (what, np.abs(post - post_x).max())


# ----------------------------------------------------------------------------------------------
# the specification, everything of one read in one forward and one backward call
# ----------------------------------------------------------------------------------------------
def oracle_all(compiled, seq, classes, max_sweeps=4096, want_cells=False):
    """dict(rc, loglike, sweeps, loglike_back, counts, post[, cells]) from oracle/forward_oracle.c; rc is OR'ed over the
    forward and the backward pass."""
    t = compiled.t
    f = util.oracle_forward(compiled, seq, want_cells=True, max_sweeps=max_sweeps)
    tok = util.tokens(seq)
    counts = np.zeros(5 + t.k + 16, dtype=np.float64)
    post = np.zeros((len(seq), len(classes)), dtype=np.float64)
    llb = C.c_double(0)
    sw = C.c_long(0)
    rc = util.forward_oracle_lib().dnab_oracle_backward_posterior(
        C.addressof(t), tok.ctypes.data, len(seq), max_sweeps, f["cells"].ctypes.data, f["loglike"], C.byref(llb),
        counts.ctypes.data, C.byref(sw), classes.encode("latin1"), len(classes), post.ctypes.data)
    out = dict(rc=rc | f["rc"], rc_forward=f["rc"], loglike=f["loglike"], sweeps=f["sweeps"], loglike_back=llb.value,
               counts=counts, post=post)
    if want_cells:
        out["cells"] = f["cells"]
    return out


def oracle_many(compiled, reads, classes, max_sweeps=4096):
    """oracle_all over many reads on every core (ctypes releases the GIL during the call)."""
    with ThreadPoolExecutor(max_workers=max(1, min(32, os.cpu_count() or 1))) as pool:
        return list(pool.map(lambda s: oracle_all(compiled, s, classes, max_sweeps), reads))


# ----------------------------------------------------------------------------------------------
# machines and reads, all seeded
# ----------------------------------------------------------------------------------------------
def _outer(symbols, seed, code_len, period):
    """An outer machine for l4c4: '^', then `period` loop states in a ring; from each, every symbol of `symbols` starts
    a seeded random code of code_len[0]..code_len[1] bits (l4c4's input) that leads to the next loop state; '$' ends
    it.  Its input symbols are '^', '$' and `symbols`."""
    rng = np.random.default_rng(seed)
    b = wide._Builder()
    s0 = b.state()
    loops = [b.state() for _ in range(period)]
    b.add(s0, loops[0], inp="^", out="^")
    for li, loop in enumerate(loops):
        for sym in symbols:
            code = "".join("01"[v] for v in rng.integers(0, 2, rng.integers(code_len[0], code_len[1] + 1)))
            prev = loop
            for j, ch in enumerate(code):
                nxt = loops[(li + 1) % period] if j == len(code) - 1 else b.state()
                b.add(prev, nxt, inp=sym if j == 0 else None, out=ch)
                prev = nxt
    end = b.state()
    b.add(loops[0], end, inp="$", out="$")
    return b.json()


# name: (outer symbols, seed, code lengths, period, states after composition onto l4c4)
COMPOSED = {
    "six_symbols": ("01CD", 1, (1, 3), 1, 451),     # 8 posterior classes: every slot of the kernel's register array
    "seven_symbols": ("01CDE", 1, (1, 2), 1, 377),  # 9 classes: refused by dnab_posterior_classes
    "w128_frontier": ("01CD", 1, (1, 3), 2, 733),   # automatic width 128 threads, >= 4 states per thread: frontier on
    "w512": ("01CD", 1, (2, 4), 6, 3236),           # automatic width 512 threads (2,048 to 4,095 states)
}
_COMPILED = {}


def compiled(name, global_=True):
    """Compiled machines by name: golden-recipe machines, k = 0 / k = 6 variants and the COMPOSED ones."""
    import dnastore_b200 as d
    key = (name, global_)
    if key not in _COMPILED:
        if name == "l4c4":
            c = util.compiled_for(("l4c4",), FLAGS, global_)
        elif name == "mr2l4c4":
            c = util.compiled_for(("l4c4", "mixradar2"), FLAGS, global_)
        elif name == "k0":
            c = util.compiled_for(("l4c4",), dict(FLAGS, length=1), global_)  # -l 1: no duplication context
        elif name == "k6":
            c = util.compiled_for(("l8c4",), dict(FLAGS, length=12), global_)  # left context 8, -l 12: k = 6 = kMaxK
        elif name in COMPOSED:
            symbols, seed, code_len, period, _ = COMPOSED[name]
            m = d.Machine.compose(d.Machine.from_json(_outer(symbols, seed, code_len, period)),
                                  d.Machine.from_file(util.machine_path("l4c4")))
            c = m.compile(util.error_flags(FLAGS, global_))
        else:
            c = wide._compiled(name, global_)
        _COMPILED[key] = c
    return _COMPILED[key]


def _walk_reads(c, n, seed, max_len=400):
    """n seeded reads of machine c: random paths to the end state, mutated with substitutions, duplications and
    deletions."""
    from benchdata import synth
    rng = np.random.default_rng(seed)
    a = c.arrays()
    out = []
    while len(out) < n:
        seq, _ = wide._walk(a, rng)
        seq = seq[:max_len]
        out.append(synth.mutate(seq, rng, sub_rate=0.02, dup_rate=0.02, max_dup=3, del_rate=0.02, max_del=3).upper())
    return out


def _indel_reads(seed=11):
    """l4c4 golden reads plus heavily mutated copies: many insertions (duplications) and deletions."""
    from benchdata import synth
    rng = np.random.default_rng(seed)
    base = [r["seq"] for r in util.golden_case("l4c4_global_mixed")["reads"]]
    return [synth.mutate(base[i], rng, sub_rate=0.03, dup_rate=0.04, max_dup=3, del_rate=0.05, max_del=4).upper()
            for i in range(len(base))]


def _golden_reads(global_=True):
    return [r["seq"] for r in util.golden_case("l4c4_global_mixed" if global_ else "l4c4_local_mixed")["reads"]]


# ----------------------------------------------------------------------------------------------
# CPU: the exact reference and the machines
# ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,global_", [("l4c4", True), ("l4c4", False), ("k0", True), ("six_symbols", False)])
def test_exact_reference_matches_linear_solve(name, global_):
    """The exact reference's log-likelihood equals test_forward.exact_forward (scipy sparse LU) to 1e-10 relative."""
    c = compiled(name, global_)
    classes = util.posterior_classes(c)
    for seq in (_golden_reads(global_)[:2] + ["", "A"]):
        ll, _, post = exact_fwdback(c, seq, classes)
        ref = exact_forward(c, seq)
        if np.isinf(ref):
            assert np.isinf(ll), (name, seq)
            continue
        assert abs(ll - ref) <= 1e-10 * max(1.0, abs(ref)), (name, seq, ll, ref)
        np.testing.assert_allclose(post.sum(axis=1), 1.0, rtol=0, atol=1e-12)  # every base is consumed exactly once


def _cases_a():
    yield "l4c4", True, _golden_reads(True)[:3] + _indel_reads()[:3]
    yield "l4c4", False, _golden_reads(False)[:3] + _indel_reads()[3:5]
    yield "mr2l4c4", False, [r["seq"] for r in util.golden_case("mr2l4c4_local")["reads"][:2]]
    yield "k0", True, _golden_reads(True)[3:5] + _indel_reads()[5:7]
    yield "six_symbols", True, _walk_reads(compiled("six_symbols", True), 3, seed=6)
    yield "six_symbols", False, _walk_reads(compiled("six_symbols", False), 2, seed=7)


@pytest.mark.parametrize("name,global_,reads", list(_cases_a()), ids=lambda v: str(v) if not isinstance(v, list) else "")
def test_exact_reference_against_specification(name, global_, reads):
    """The specification's log-likelihood, counts and posteriors against the exact reference, within the calibrated
    bounds (LL_TOL, COUNT_TOL, POST_TOL); the posterior and the counts also agree with each other."""
    c = compiled(name, global_)
    classes = util.posterior_classes(c)
    k = c.t.k
    for seq in reads:
        o = oracle_all(c, seq, classes)
        assert o["rc"] == 0
        assert_near_exact(exact_fwdback(c, seq, classes), o["loglike"], o["counts"], o["post"], (name, global_, seq))
        assert abs(o["post"][:, :-1].sum() - o["counts"][2]) < 1e-9 * max(1.0, o["counts"][2])
        assert abs(o["post"].sum() - o["counts"][5 + k:].sum()) < 1e-9 * max(1, len(seq))


def test_exact_comparison_rejects_wrong_counts_and_posteriors():
    """The exact comparison is sharp enough to catch a count filed in the wrong slot or a posterior one base off."""
    c = compiled("l4c4", True)
    classes = util.posterior_classes(c)
    seq = _indel_reads()[0]
    o = oracle_all(c, seq, classes)
    exact = exact_fwdback(c, seq, classes)
    assert_near_exact(exact, o["loglike"], o["counts"], o["post"], "as computed")
    swapped = o["counts"].copy()
    swapped[[0, 3]] = swapped[[3, 0]]  # nDelOpen <-> nDelExtend
    with pytest.raises(AssertionError):
        assert_near_exact(exact, o["loglike"], swapped, None, "nDelOpen and nDelExtend swapped")
    k = c.t.k
    sub = o["counts"].copy()
    sub[5 + k:] = sub[5 + k:].reshape(4, 4).T.ravel()  # nSub with machine and read base exchanged
    with pytest.raises(AssertionError):
        assert_near_exact(exact, o["loglike"], sub, None, "nSub transposed")
    with pytest.raises(AssertionError):
        assert_near_exact(exact, o["loglike"], None, np.roll(o["post"], 1, axis=0), "posterior rows shifted by one base")
    with pytest.raises(AssertionError):
        assert_near_exact(exact, o["loglike"] - 3 * LL_TOL, None, None, "log-likelihood too low")


@pytest.mark.parametrize("name", list(COMPOSED))
def test_composed_machines(name):
    """The generated machines have the state counts (hence the automatic CTA widths) and class counts the GPU tests rely
    on."""
    c = compiled(name)
    assert c.t.n_states == COMPOSED[name][4]
    assert len(util.posterior_classes(c)) == len(COMPOSED[name][0]) + 4  # '-', '^', '$', '+'


def test_k_machines():
    assert compiled("k0").t.k == 0 and compiled("k6").t.k == 6 and compiled("l4c4").t.k == 2


# ----------------------------------------------------------------------------------------------
# GPU
# ----------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def d():
    import dnastore_b200
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return dnastore_b200


def _sm_count():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _auto_threads(n_states):
    return 1024 if n_states >= 4096 else 512 if n_states >= 2048 else 256 if n_states >= 1024 else 128


def _run_all(dec, reads, max_sweeps=0, want_cells=False):
    """forward, fwdback_counts and posterior of one batch, each with the launch shape it used."""
    out = {}
    out["fwd"] = dec.forward(reads, max_sweeps=max_sweeps, want_cells=want_cells)
    st = dec.stats()
    out["fwd_shape"] = (st["last_fwd_threads"], st["last_fwd_blocks"])
    out["fb"] = dec.fwdback_counts(reads, max_sweeps=max_sweeps)
    st = dec.stats()
    out["fb_shape"] = (st["last_fwd_threads"], st["last_fwd_blocks"])
    out["post"] = dec.posterior(reads, max_sweeps=max_sweeps)
    st = dec.stats()
    out["post_shape"] = (st["last_fwd_threads"], st["last_fwd_blocks"])
    return out


def _check_oracle(got, reads, oracle, what, cells_of_read0=None):
    """Every read of a _run_all result against oracle_all results: log-likelihoods bit for bit, sweeps and status
    exactly, counts and posteriors to 1e-9, the decoded string = the argmax of the posterior."""
    f, fb, p = got["fwd"], got["fb"], got["post"]
    classes = p["classes"]
    for i, o in enumerate(oracle):
        w = (what, i, len(reads[i]))
        assert util.hexf(f["loglike"][i]) == util.hexf(o["loglike"]), w
        assert f["sweeps"][i] == o["sweeps"] and f["status"][i] == o["rc_forward"], w
        assert util.hexf(fb["loglike"][i]) == util.hexf(o["loglike"]), w
        assert util.hexf(fb["loglike_back"][i]) == util.hexf(o["loglike_back"]), w
        assert fb["status"][i] == o["rc"] and p["status"][i] == o["rc"], w
        np.testing.assert_allclose(fb["counts"][i], o["counts"], rtol=1e-9, atol=1e-12, err_msg=str(w))
        assert util.hexf(p["loglike"][i]) == util.hexf(o["loglike"]), w
        np.testing.assert_allclose(p["post"][i], o["post"], rtol=1e-9, atol=1e-12, err_msg=str(w))
        assert p["decoded"][i] == "".join(classes[j] for j in p["post"][i].argmax(axis=1)), w
    if cells_of_read0 is not None:
        assert f["cells"].tobytes() == cells_of_read0.tobytes(), what


def _check_invariants(got, reads, k, local, n_states, what):
    """What holds for every read whatever the reference: backward = forward log-likelihood up to the table
    log_sum_exp, every base consumed once (sum of nSub = L, posterior rows sum to 1), every deletion that opens ends,
    nTanDup = sum of nLen, and the posterior binned by class = nNoGap.
    In local mode the likelihood is a table log-sum over every state, whose error grows with the state count N: the
    nSub sum of a 1-base read is 1.0011 on l4c4 (384 states), 1.0066 on the 3,236-state machine of (d) (whose
    specification is there 6.6e-3 below the exact log-likelihood) and 1.0214 on l8c4 -l 12 (10,746 states), about
    2e-6 * N; on the latter backward and forward differ by up to 1.2e-2.  So local mode gets 2e-3 + 5e-6 * N."""
    fb, p = got["fb"], got["post"]
    tol = 2e-3 + (5e-6 * n_states if local else 0.)
    for i, seq in enumerate(reads):
        w = (what, i, len(seq))
        c = fb["counts"][i]
        assert fb["status"][i] == 0 and p["status"][i] == 0, w
        assert abs(fb["loglike_back"][i] - fb["loglike"][i]) < tol, w
        assert abs(c[5 + k:].sum() - len(seq)) < tol * max(1, len(seq)), w
        assert abs(c[0] - c[4]) < 1e-3 * max(1.0, c[0]), w
        assert abs(c[1] - c[5:5 + k].sum()) < 1e-12 * max(1.0, c[1]), w
        if len(seq):
            np.testing.assert_allclose(p["post"][i].sum(axis=1), 1.0, atol=max(tol, 3e-3), err_msg=str(w))
            assert abs(p["post"][i][:, :-1].sum() - c[2]) < 1e-9 * max(1.0, c[2]), w


def _same_bits(a, b, what, counts_exact=True):
    """Two _run_all results of the same reads: the log-likelihoods, sweeps and status bit for bit; counts and
    posteriors bit for bit too when both ran at the same CTA width (the state sums then run in the same order),
    else within 1e-9."""
    for key in ("loglike", "sweeps", "status"):
        assert a["fwd"][key].tobytes() == b["fwd"][key].tobytes(), (what, "forward", key)
    for key in ("loglike", "loglike_back", "status"):
        assert a["fb"][key].tobytes() == b["fb"][key].tobytes(), (what, "fwdback", key)
    assert a["post"]["loglike"].tobytes() == b["post"]["loglike"].tobytes(), what
    if counts_exact:
        assert a["fb"]["counts"].tobytes() == b["fb"]["counts"].tobytes(), (what, "counts")
        assert all(x.tobytes() == y.tobytes() for x, y in zip(a["post"]["post"], b["post"]["post"])), (what, "posterior")
        assert a["post"]["decoded"] == b["post"]["decoded"], what
    else:
        np.testing.assert_allclose(a["fb"]["counts"], b["fb"]["counts"], rtol=1e-9, atol=1e-12, err_msg=str(what))
        for x, y in zip(a["post"]["post"], b["post"]["post"]):
            np.testing.assert_allclose(x, y, rtol=1e-9, atol=1e-12, err_msg=str(what))


# (b) every CTA width and grid cap on l4c4 -------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("global_", [True, False], ids=["global", "local"])
def test_gpu_every_width_and_cap(d, global_):
    """fwd_threads in {32, 64, 96, 128, 512, 1024} x fwd_blocks in {0, 1, 7} on l4c4 (384 states: 32 and 64 threads
    turn the frontier on, 1024 leave most lanes idle, 1 and 7 CTAs take many reads each): the same bits as the
    automatic shape and as the specification."""
    c = compiled("l4c4", global_)
    reads = _golden_reads(global_) + ["", "A", "GT", "ACG", "TTAC"] + _indel_reads()[:6]
    dec = d.Decoder(c, device=0)
    classes = dec.posterior_classes()
    oracle = oracle_many(c, reads, classes)
    auto = _run_all(dec, reads, want_cells=True)
    assert auto["fwd_shape"] == auto["fb_shape"] == auto["post_shape"] == (128, len(reads))
    _check_oracle(auto, reads, oracle, "auto", oracle_all(c, reads[0], classes, want_cells=True)["cells"])
    sm = _sm_count()
    for threads in (32, 64, 96, 128, 512, 1024):
        for blocks in (0, 1, 7):
            dec.set_option("fwd_threads", threads)
            dec.set_option("fwd_blocks", blocks)
            got = _run_all(dec, reads, want_cells=True)
            want = min(len(reads), sm * (1024 // threads), blocks or len(reads))
            what = (global_, threads, blocks)
            assert got["fwd_shape"] == got["fb_shape"] == got["post_shape"] == (threads, want), (what, got["fwd_shape"])
            _same_bits(got, auto, what, counts_exact=threads == 128)
            assert got["fwd"]["cells"].tobytes() == auto["fwd"]["cells"].tobytes(), what
            if threads != 128:
                _check_oracle(got, reads, oracle, what)
    dec.set_option("fwd_threads", 0)
    dec.set_option("fwd_blocks", 0)
    _same_bits(_run_all(dec, reads), auto, "automatic again")
    assert dec.stats()["last_fwd_threads"] == 128


@pytest.mark.gpu
def test_gpu_schedule_options_refuse_bad_values(d):
    dec = d.Decoder(compiled("l4c4"), device=0)
    for bad in (1, 16, 33, 100, 1025, 2048):
        with pytest.raises(d.DnabError) as e:
            dec.set_option("fwd_threads", bad)
        assert e.value.code == -1 and "fwd_threads" in str(e.value)
    with pytest.raises(d.DnabError):
        dec.set_option("fwd_blocks", 1 << 32)
    out = dec.forward(["ACGT"])
    assert dec.stats()["last_fwd_threads"] == 128
    assert util.hexf(out["loglike"][0]) == util.hexf(util.oracle_forward(compiled("l4c4"), "ACGT")["loglike"])


# (c) many reads per CTA with the automatic shape, (j) invariants ---------------------------------------
@pytest.mark.gpu
def test_gpu_many_reads_per_cta_l4c4(d):
    """About 3,000 seeded l4c4 reads (more than the 1,184 CTAs of the automatic shape), with the empty read, 1 to 4
    bases and full-length reads in shuffled order: every read against the specification, the cells of read 0, and the
    invariants."""
    from benchdata import synth
    c = compiled("l4c4")
    rng = np.random.default_rng(3000)
    base = _golden_reads(True)
    reads = [synth.mutate(base[i % len(base)], rng, sub_rate=0.02, dup_rate=0.01, max_dup=2, del_rate=0.01, max_del=3).upper()
             for i in range(2980)]
    reads += ["", "", "A", "C", "GT", "TA", "ACG", "TTT", "ACGT", "GATC"] + base[:10]
    order = rng.permutation(len(reads))
    reads = [reads[i] for i in order]
    dec = d.Decoder(c, device=0)
    classes = dec.posterior_classes()
    got = _run_all(dec, reads, want_cells=True)
    assert got["fwd_shape"] == (128, min(len(reads), 8 * _sm_count())) and len(reads) > 8 * _sm_count()
    oracle = oracle_many(c, reads, classes)
    cells0 = oracle_all(c, reads[0], classes, want_cells=True)["cells"]
    _check_oracle(got, reads, oracle, "l4c4 x 3000", cells0)
    _check_invariants(got, reads, c.t.k, c.t.local, c.t.n_states, "l4c4 x 3000")


@pytest.mark.gpu
def test_gpu_many_reads_per_cta_cfg5(d):
    """About 400 cfg5 reads (l8c4, 10,746 states, 148 CTAs of 1,024 threads): every read bit-identical to the same read
    run in chunks of at most 148 reads (one read per CTA); a seeded sample, cut to 30 bases in the batch itself,
    against the specification."""
    from benchdata import synth
    c = util.machine_from_recipe(("l8c4",)).compile(d.ErrorFlags(length=8, global_=True))
    pool = synth.load_pool("cfg5_l8c4_150b")
    reads = list(synth.mutate_subs_batch([pool[i % len(pool)] for i in range(400)], np.random.default_rng(5), sub_rate=0.01))
    rng = np.random.default_rng(55)
    sample = sorted(rng.choice(len(reads), 6, replace=False).tolist())
    for i in sample:
        reads[i] = reads[i][:30]
    dec = d.Decoder(c, device=0)
    classes = dec.posterior_classes()
    whole = _run_all(dec, reads)
    assert whole["fwd_shape"] == (1024, _sm_count())
    chunk = _sm_count()
    parts = [_run_all(dec, reads[i:i + chunk]) for i in range(0, len(reads), chunk)]
    for key in ("loglike", "sweeps", "status"):
        assert whole["fwd"][key].tobytes() == np.concatenate([p["fwd"][key] for p in parts]).tobytes(), key
    for key in ("loglike", "loglike_back", "counts", "status"):
        assert whole["fb"][key].tobytes() == np.concatenate([p["fb"][key] for p in parts]).tobytes(), key
    assert whole["post"]["loglike"].tobytes() == np.concatenate([p["post"]["loglike"] for p in parts]).tobytes()
    assert all(x.tobytes() == y.tobytes() for x, y in zip(whole["post"]["post"], [r for p in parts for r in p["post"]["post"]]))
    assert whole["post"]["decoded"] == [r for p in parts for r in p["post"]["decoded"]]
    oracle = oracle_many(c, [reads[i] for i in sample], classes)
    sub = {"fwd": {k: v[sample] for k, v in whole["fwd"].items()}, "fb": {k: v[sample] for k, v in whole["fb"].items()},
           "post": dict(classes=classes, loglike=whole["post"]["loglike"][sample], status=whole["post"]["status"][sample],
                        post=[whole["post"]["post"][i] for i in sample], decoded=[whole["post"]["decoded"][i] for i in sample])}
    _check_oracle(sub, [reads[i] for i in sample], oracle, "cfg5 sample")
    _check_invariants(whole, reads, c.t.k, c.t.local, c.t.n_states, "cfg5 x 400")


# (d) the automatic widths the golden machines miss -------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("global_", [True, False], ids=["global", "local"])
@pytest.mark.parametrize("name,threads", [("w128_frontier", 128), ("w512", 512)])
def test_gpu_automatic_widths(d, name, threads, global_):
    """733 states (128 threads, frontier on) and 3,236 states (512 threads): against the specification, and the smaller
    machine also against the exact reference."""
    c = compiled(name, global_)
    assert c.t.n_states == COMPOSED[name][4] and _auto_threads(c.t.n_states) == threads
    reads = _walk_reads(c, 40, seed=COMPOSED[name][4] + global_, max_len=120) + ["", "A"]
    dec = d.Decoder(c, device=0)
    classes = dec.posterior_classes()
    got = _run_all(dec, reads)
    assert got["fwd_shape"][0] == got["fb_shape"][0] == threads
    _check_oracle(got, reads, oracle_many(c, reads, classes), (name, global_))
    _check_invariants(got, reads, c.t.k, c.t.local, c.t.n_states, (name, global_))
    if c.t.n_states <= 1500:
        for i in (0, 1):
            assert_near_exact(exact_fwdback(c, reads[i], classes), got["fb"]["loglike"][i], got["fb"]["counts"][i],
                              got["post"]["post"][i], (name, global_, i))


# (e) the sweep limit ------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("threads", [0, 32], ids=["auto", "frontier"])
@pytest.mark.parametrize("global_", [True, False], ids=["global", "local"])
def test_gpu_sweep_limit(d, global_, threads):
    """max_sweeps 1, 2, 3: status 1 and the specification's bits at the same limit (full sweeps at 128 threads, the
    frontier at 32)."""
    c = compiled("l4c4", global_)
    reads = _golden_reads(global_)[:6] + _indel_reads()[:4]
    dec = d.Decoder(c, device=0)
    dec.set_option("fwd_threads", threads)
    classes = dec.posterior_classes()
    for max_sweeps in (1, 2, 3):
        got = _run_all(dec, reads, max_sweeps=max_sweeps)
        oracle = oracle_many(c, reads, classes, max_sweeps=max_sweeps)
        assert all(o["rc"] == 1 for o in oracle)
        assert (got["fwd"]["status"] == 1).all() and (got["fb"]["status"] == 1).all() and (got["post"]["status"] == 1).all()
        _check_oracle(got, reads, oracle, (global_, threads, max_sweeps))


# (f) duplication depth k = 0 and k = 6 --------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("global_", [True, False], ids=["global", "local"])
@pytest.mark.parametrize("name", ["k0", "k6"])
def test_gpu_duplication_depth(d, name, global_):
    """k = 0 (no T planes, counts of length 21) on l4c4 -l 1, also against the exact reference; k = 6 (every T plane,
    counts of length 27) on l8c4 -l 12 with short reads."""
    c = compiled(name, global_)
    k = c.t.k
    assert k == (0 if name == "k0" else 6)
    if name == "k0":
        reads = _golden_reads(global_)[:6] + _indel_reads()[:4] + ["", "A"]
    else:
        reads = [s[:n] for s, n in zip([r["seq"] for r in util.golden_case("cfg5_l8_global")["reads"]] * 2, (30, 24, 28, 20, 16, 12, 8, 4))]
        reads += ["", "A", "GATTACA"]
    dec = d.Decoder(c, device=0)
    classes = dec.posterior_classes()
    got = _run_all(dec, reads)
    assert got["fb"]["counts"].shape == (len(reads), 5 + k + 16)
    _check_oracle(got, reads, oracle_many(c, reads, classes), (name, global_))
    _check_invariants(got, reads, k, c.t.local, c.t.n_states, (name, global_))
    if name == "k0":
        for i in (0, 7):
            assert_near_exact(exact_fwdback(c, reads[i], classes), got["fb"]["loglike"][i], got["fb"]["counts"][i],
                              got["post"]["post"][i], (name, global_, i))


# (g) high-degree machines, (j) invariants -------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("global_", [True, False], ids=["global", "local"])
@pytest.mark.parametrize("name", wide.MACHINES)
def test_gpu_high_degree_machines(d, name, global_):
    """The four machines of test_gpu_wide_states (hubs of 300 to 1,200 in- or out-transitions, walked by the frontier's
    pass A and the evaluate2 loops): all 48 reads against the invariants, the first reads against the specification."""
    c = compiled(name, global_)
    reads = wide._reads(name)
    n_oracle = 4 if name == "d_selector_l4c4" else 16
    dec = d.Decoder(c, device=0)
    classes = dec.posterior_classes()
    got = _run_all(dec, reads)
    assert got["fwd_shape"][0] == _auto_threads(c.t.n_states)
    sub = {"fwd": {k: v[:n_oracle] for k, v in got["fwd"].items()}, "fb": {k: v[:n_oracle] for k, v in got["fb"].items()},
           "post": dict(got["post"], loglike=got["post"]["loglike"][:n_oracle], status=got["post"]["status"][:n_oracle])}
    _check_oracle(sub, reads[:n_oracle], oracle_many(c, reads[:n_oracle], classes), (name, global_))
    _check_invariants(got, reads, c.t.k, c.t.local, c.t.n_states, (name, global_))


# (h) long reads --------------------------------------------------------------------------------------------------
def _long_read(c, n, seed):
    """n bases from a seeded random walk through machine c (taking any transition; no need to reach the end), with 1%
    substitutions."""
    a = c.arrays()
    rng = np.random.default_rng(seed)
    outs = [[] for _ in range(a["n_states"])]
    for dst in range(a["n_states"]):
        for e in range(a["emit_off"][dst], a["emit_off"][dst + 1]):
            outs[a["emit_src"][e]].append((dst, int(a["emit_base"][e])))
        for e in range(a["null_off"][dst], a["null_off"][dst + 1]):
            outs[a["null_src"][e]].append((dst, None))
    s, seq = 0, []
    while len(seq) < n:
        if not outs[s]:
            s = 0
            continue
        s, b = outs[s][rng.integers(len(outs[s]))]
        if b is not None:
            seq.append(b if rng.random() > 0.01 else int(rng.integers(4)))
    return "".join("ACGT"[b] for b in seq)


@pytest.mark.gpu
def test_gpu_long_reads(d):
    """Two reads of exactly 16,000 bases (the longest accepted) batched with short reads through one CTA; a read of
    16,001 bases is refused and the handle still gives the same bits afterwards."""
    c = compiled("l4c4")
    reads = ["ACGT", _long_read(c, 16000, 1), "", _long_read(c, 16000, 2), _golden_reads()[0]]
    dec = d.Decoder(c, device=0)
    dec.set_option("fwd_blocks", 1)
    classes = dec.posterior_classes()
    fwd = dec.forward(reads)
    assert (dec.stats()["last_fwd_threads"], dec.stats()["last_fwd_blocks"]) == (128, 1)
    fb = dec.fwdback_counts(reads)
    oracle = oracle_many(c, reads, classes)
    for i, o in enumerate(oracle):
        assert util.hexf(fwd["loglike"][i]) == util.hexf(o["loglike"]) and fwd["sweeps"][i] == o["sweeps"], i
        assert fwd["status"][i] == 0 and fb["status"][i] == 0, i
        assert util.hexf(fb["loglike"][i]) == util.hexf(o["loglike"]), i
        assert util.hexf(fb["loglike_back"][i]) == util.hexf(o["loglike_back"]), i
        np.testing.assert_allclose(fb["counts"][i], o["counts"], rtol=1e-9, atol=1e-12, err_msg=str(i))
    too_long = reads[1] + "A"
    for call in (dec.forward, dec.fwdback_counts, dec.posterior):
        with pytest.raises(d.DnabError, match="longer than 16000") as e:
            call(["ACGT", too_long])
        assert e.value.code == -1
    fwd2, fb2 = dec.forward(reads), dec.fwdback_counts(reads)
    for key in fwd:
        assert fwd[key].tobytes() == fwd2[key].tobytes(), key
    for key in fb:
        assert fb[key].tobytes() == fb2[key].tobytes(), key


# (i) posterior classes at the limit ---------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("global_", [True, False], ids=["global", "local"])
def test_gpu_eight_posterior_classes(d, global_):
    """A machine with 6 input symbols has 8 classes, every slot of the kernel's register array: against the
    specification and the exact reference."""
    c = compiled("six_symbols", global_)
    dec = d.Decoder(c, device=0)
    classes = dec.posterior_classes()
    assert len(classes) == 8 and classes == util.posterior_classes(c)
    reads = _walk_reads(c, 24, seed=8 + global_) + ["", "T"]
    got = _run_all(dec, reads)
    _check_oracle(got, reads, oracle_many(c, reads, classes), ("six_symbols", global_))
    _check_invariants(got, reads, c.t.k, c.t.local, c.t.n_states, ("six_symbols", global_))
    for i in (0, 1):
        assert_near_exact(exact_fwdback(c, reads[i], classes), got["fb"]["loglike"][i], got["fb"]["counts"][i],
                          got["post"]["post"][i], ("six_symbols", global_, i))
    used = np.concatenate(got["post"]["post"][:24]).max(axis=0)
    assert (used[1:] > 0).all(), used  # every input symbol's class and "+" take part


@pytest.mark.gpu
def test_gpu_seven_input_symbols_refused(d):
    """7 input symbols would need 9 classes: refused with a message that names the limit (6) and the machine's count
    (7); forward on the same handle still works."""
    c = compiled("seven_symbols")
    dec = d.Decoder(c, device=0)
    for call in (dec.posterior_classes, lambda: dec.posterior(["ACGT"])):
        with pytest.raises(d.DnabError, match=r"at most 6 input symbols apart; this machine has 7") as e:
            call()
        assert e.value.code == -1
    reads = _walk_reads(c, 4, seed=9)
    out = dec.forward(reads)
    for i, s in enumerate(reads):
        assert util.hexf(out["loglike"][i]) == util.hexf(util.oracle_forward(c, s)["loglike"]), i
