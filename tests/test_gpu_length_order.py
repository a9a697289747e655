"""GPU (B200): the read-batched kernel forms its groups of 32 reads by length (descending, ties in input order) on the
device, from the device-resident lengths, for the host-buffer and the device-pointer entries alike.  A read left out
of the order, or dealt twice, would leave an output untouched or overwritten; the one-read-per-cluster push kernel,
which forms no groups, is the reference."""
import numpy as np
import pytest

import dnab_testutil as util

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def d():
    import dnastore_b200
    return dnastore_b200


@pytest.mark.parametrize("slack", [0, 2800])  # max_read_len above the longest read: more length bins than threads
@pytest.mark.parametrize("n", [33, 517])
def test_gpu_length_groups_same_results_on_both_entries(d, n, slack):
    import torch

    import bench
    w = bench.WORKLOADS["cfg1"]
    compiled = util.machine_from_recipe(w["recipe"]).compile(d.ErrorFlags(length=w["length"], global_=True))
    rng = np.random.default_rng(n)
    # ragged lengths with many ties; a trimmed read may have no decoding at all, which must come out the same too
    reads = [r[:len(r) - int(rng.integers(0, 41))] for r in bench.make_reads(w, n, seed=4243)]

    ref = d.Decoder(compiled, device=0)
    ref.set_option("kernel", 2)
    want = ref.viterbi(reads)

    dec = d.Decoder(compiled, device=0)
    dec.set_option("kernel", 1)
    got = dec.viterbi(reads)
    assert dec.batch_info()["enabled"]
    assert got["loglike"].tobytes() == want["loglike"].tobytes()
    assert got["decoded"] == want["decoded"]
    assert got["status"].tolist() == want["status"].tolist()

    packed, byte_off, read_len = d.pack_reads(reads)
    max_len = int(read_len.max()) + slack
    stride = 2 * max_len + 64
    dev = torch.device("cuda", 0)
    p, o, ln = (torch.from_numpy(np.ascontiguousarray(a)).to(dev) for a in (packed, byte_off, read_len))
    ll = torch.full((n,), float("nan"), dtype=torch.float64, device=dev)
    raw = torch.zeros(n * stride, dtype=torch.uint8, device=dev)
    dl = torch.full((n,), -1, dtype=torch.int32, device=dev)
    status = torch.full((n,), -1, dtype=torch.int32, device=dev)
    dec.viterbi_device(n, max_len, p.data_ptr(), o.data_ptr(), ln.data_ptr(), ll.data_ptr(), raw.data_ptr(), stride,
                       dl.data_ptr(), status.data_ptr(), torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    ll, raw, dl, status = ll.cpu().numpy(), raw.cpu().numpy().reshape(n, stride), dl.cpu().numpy(), status.cpu().numpy()
    assert ll.tobytes() == want["loglike"].tobytes()
    assert status.tolist() == want["status"].tolist()
    assert [bytes(raw[i, :dl[i]]).decode("latin1") for i in range(n)] == want["decoded"]
