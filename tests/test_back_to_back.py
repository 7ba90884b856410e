"""Back-to-back capture decodes on one stream (run with -m gpu on a B200).

rx_pack_kernel is launched with programmatic dependent launch: a launch may start while the previous one still runs, and
only waits for it before it stores outputs.  These tests check that such a sequence decodes exactly as the same calls made
one at a time, that a shared output buffer ends up holding the last call's records, that ordinary kernels before and after
a decode still see its inputs and outputs in order, and what rfid_b200_kernel_time reports for such a sequence.
"""
import numpy as np
import pytest

from conftest import records_equal
from gen2_uhf_rfid_reader_b200 import synth

pytestmark = pytest.mark.gpu

NSEG = 1000          # bench.py cfg2: 143 CTAs of 7 segments, one CTA per SM
MAXW = 4
K = 6


@pytest.fixture(scope="module")
def rx():
    from gen2_uhf_rfid_reader_b200 import capi
    return capi.Gen2Rx()


@pytest.fixture(scope="module")
def caps():
    """two captures of NSEG segments with the same segment table (as bench.py cfg2's)"""
    import torch
    from gen2_uhf_rfid_reader_b200 import capi
    dev = torch.device("cuda:0")
    cs = [synth.make_capture(NSEG, seed=1234 + 17 * b, device=dev) for b in range(2)]
    assert all((c["segments"] == cs[0]["segments"]).all() for c in cs)
    return [c["iq"] for c in cs], capi.segments_to_device(cs[0]["segments"], dev)


def _buffers(dev):
    import torch
    return torch.zeros((NSEG * MAXW, 64), dtype=torch.uint8, device=dev), torch.zeros(NSEG, dtype=torch.int32, device=dev)


@pytest.fixture(scope="module")
def one_at_a_time(rx, caps):
    """records and counts of each capture, decoded alone with a synchronise after the call"""
    import torch
    from gen2_uhf_rfid_reader_b200 import capi
    iqs, segs = caps
    out = []
    for iq in iqs:
        res, cnt = _buffers(iq.device)
        rx.decode_capture(iq, segs, MAXW, res, cnt)
        torch.cuda.synchronize()
        out.append(capi.results_to_numpy(res, cnt, MAXW))
    assert all(int(c.sum()) > 0 for _, c in out)
    return out


def _stream(kind, dev):
    import torch
    s = torch.cuda.default_stream(dev) if kind == "default" else torch.cuda.Stream(device=dev)
    assert (s.cuda_stream == 0) == (kind == "default")
    return s


@pytest.mark.parametrize("stream_kind", ["default", "created"])
def test_back_to_back_distinct_buffers(rx, caps, one_at_a_time, stream_kind):
    """K decodes of alternating captures with no synchronisation in between, each into its own buffers: every call's
    records bit-identical to the same call made alone"""
    import torch
    from gen2_uhf_rfid_reader_b200 import capi
    iqs, segs = caps
    s = _stream(stream_kind, iqs[0].device)
    bufs = [_buffers(iqs[0].device) for _ in range(K)]
    torch.cuda.synchronize()
    for k in range(K):
        rx.decode_capture(iqs[k % 2], segs, MAXW, bufs[k][0], bufs[k][1], stream=s)
    torch.cuda.synchronize()
    for k in range(K):
        recs, counts = capi.results_to_numpy(bufs[k][0], bufs[k][1], MAXW)
        ref_recs, ref_counts = one_at_a_time[k % 2]
        assert counts.tolist() == ref_counts.tolist(), "call %d" % k
        bad = records_equal(recs, ref_recs)
        assert not bad, "call %d: fields differ: %s" % (k, bad)


@pytest.mark.parametrize("stream_kind", ["default", "created"])
def test_back_to_back_shared_buffer(rx, caps, one_at_a_time, stream_kind):
    """K decodes of alternating captures into ONE result / count buffer: after the final synchronise it holds the last
    call's counts and, in every slot that call stored, its records (a launch stores only after the previous one is done)"""
    import torch
    from gen2_uhf_rfid_reader_b200 import capi
    iqs, segs = caps
    s = _stream(stream_kind, iqs[0].device)
    res, cnt = _buffers(iqs[0].device)
    torch.cuda.synchronize()
    for k in range(K):
        rx.decode_capture(iqs[k % 2], segs, MAXW, res, cnt, stream=s)
    torch.cuda.synchronize()
    recs, counts = capi.results_to_numpy(res, cnt, MAXW)
    ref_recs, ref_counts = one_at_a_time[(K - 1) % 2]
    assert counts.tolist() == ref_counts.tolist()
    stored = np.arange(MAXW)[None, :] < np.minimum(ref_counts, MAXW)[:, None]
    bad = records_equal(recs[stored], ref_recs[stored])
    assert not bad, "fields differ: %s" % bad


def test_ordering_with_ordinary_kernels(rx, oracle):
    """a torch kernel writes the capture, the decode reads it, a torch kernel reads the records, and the next round
    rewrites the same capture buffer -- no synchronisation anywhere: every round's records equal the oracle's"""
    import torch
    from gen2_uhf_rfid_reader_b200 import capi
    dev = torch.device("cuda:0")
    cs = [synth.make_capture(300, seed=71 + b) for b in range(2)]
    assert (cs[0]["segments"] == cs[1]["segments"]).all()
    srcs = [c["iq"].to(dev).view(torch.float32) for c in cs]
    segs = capi.segments_to_device(cs[0]["segments"], dev)
    iq = torch.empty_like(srcs[0])
    res = torch.zeros((300 * MAXW, 64), dtype=torch.uint8, device=dev)
    cnt = torch.zeros(300, dtype=torch.int32, device=dev)
    torch.cuda.synchronize()
    outs = []
    for k in range(4):
        torch.mul(srcs[k % 2], 1.0, out=iq)            # x * 1 is exact for every float, signed zeros included
        rx.decode_capture(iq, segs, MAXW, res, cnt)
        outs.append((res.to(torch.int16), cnt + 0))
    torch.cuda.synchronize()
    for b in range(2):
        orecs, ocounts, _ = oracle.decode_segments(cs[b]["iq"].numpy(), cs[b]["segments"], max_per_seg=MAXW)
        for k in range(b, 4, 2):
            recs, counts = capi.results_to_numpy(outs[k][0].to(torch.uint8), outs[k][1], MAXW)
            assert counts.tolist() == ocounts.tolist(), "round %d" % k
            bad = records_equal(recs, orecs)
            assert not bad, "round %d: fields differ: %s" % (k, bad)


@pytest.mark.parametrize("n", [8, 300])   # 300: more launches than the context's timing slots, drained on the way
def test_kernel_time_back_to_back(rx, caps, n):
    """kernel_time over n back-to-back launches counts n launches, a positive time each, and no more device time in
    total than CUDA events around the whole sequence"""
    import torch
    iqs, segs = caps
    res, cnt = _buffers(iqs[0].device)
    s = torch.cuda.current_stream(iqs[0].device)
    torch.cuda.synchronize()
    rx.enable_kernel_timing(True)
    rx.kernel_time(reset=True)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(s)
    for k in range(n):
        rx.decode_capture(iqs[k % 2], segs, MAXW, res, cnt, stream=s)
    ev1.record(s)
    torch.cuda.synchronize()
    ms, launches = rx.kernel_time(reset=True)
    rx.enable_kernel_timing(False)
    assert launches == n
    assert ms > 0 and ms / n > 0.005
    assert ms <= ev0.elapsed_time(ev1)
    assert rx.kernel_time(reset=True) == (0.0, 0)
