"""GPU (B200): a decoder handle keeps a consistent launch plan when a new plan cannot be made.

The push kernel plans for the longest read seen so far; a longer read makes the handle plan again. When that
fails, the handle must go on decoding with the plan it had, not with a mix of the old plan and new tables.
"""
import pytest

import dnab_testutil as util

pytestmark = pytest.mark.gpu


def test_gpu_failed_replan_keeps_the_working_plan():
    import dnastore_b200 as d
    case = util.golden_case("l4c4_global_mixed")
    dec = d.Decoder(util.compiled_for_case(case), device=0)
    # the push kernel: the read-batched kernel's layout does not depend on the read length, so it would take the long read
    dec.set_option("kernel", 2)
    reads = [r["seq"] for r in case["reads"]]
    before = dec.viterbi(reads, want_path=True)
    info = dec.info()
    # the packed sequence of a read is staged in shared memory: 1.2 M bases (300 KB) fit no CTA of any cluster
    with pytest.raises(d.DnabError, match="does not fit"):
        dec.viterbi(["ACGT" * 300_000])
    assert dec.info() == info
    after = dec.viterbi(reads, want_path=True)
    assert after["loglike"].tobytes() == before["loglike"].tobytes()
    assert after["decoded"] == before["decoded"]
    assert (after["status"] == before["status"]).all()
    assert all(x.tolist() == y.tolist() for x, y in zip(after["path"], before["path"]))
    for i, r in enumerate(case["reads"]):
        assert after["decoded"][i] == r["decoded"], r["name"]
        assert util.hexf(after["loglike"][i]) == util.hexf(r["loglike_hex"]), r["name"]
