"""GPU parity tests (run with -m gpu on a B200): the CUDA path, called through the C-ABI, against the oracle.

Bar: bit-exact for every field of every record -- decoded RN16/EPC bits, CRC flags, sync indices, window
positions, and also the float outputs (correlation score, channel estimate, T), which the north star only
asks to match within 1e-5 relative.
"""
import json
import os

import numpy as np
import pytest

from conftest import GOLDEN, load_json, records_equal, ref_segments
from gen2_uhf_rfid_reader_b200 import abi, synth

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def rx():
    from gen2_uhf_rfid_reader_b200 import capi
    return capi.Gen2Rx()


def _assert_same(got, ref, what=""):
    bad = records_equal(got, ref)
    assert not bad, "%s fields differ: %s" % (what, bad)


# ------------------------------------------------------------------ cfg1: the reference's own recording
def _assert_reference_stats(st, g):
    """READER_STATS of a continuous decode against the reference's run on the same capture"""
    assert (st.n_queries_sent, st.cur_inventory_round, st.cur_slot_number, st.n_epc_correct) == \
        (g["n_queries_sent"], g["cur_inventory_round"], g["cur_slot_number"], g["n_epc_correct"])
    assert st.tag_map() == {int(k): v for k, v in g["tag_reads"].items()}


def test_cfg1_capture_bit_exact_and_readme_stats(rx, cfg1_iq, cfg1_golden, cfg1_head_stats):
    """BASELINE.json configs[0]: misc/data/file_source_test (its first 15 rounds), FIXED_Q=0, as one continuous
    segment; stats as the reference's print_results on the same samples (README.md:48-53 for the whole file)"""
    recs, counts = rx.decode_capture_host(cfg1_iq, abi.make_segments([0], [cfg1_iq.size]), max_windows=256)
    assert counts[0] == 31
    _assert_same(recs[0, :31], cfg1_golden, "cfg1")
    rel = np.abs(recs[0, :31]["score"] - cfg1_golden["score"]) / cfg1_golden["score"]
    assert rel.max() <= 1e-5   # north-star tolerance (actually 0)
    st = rx.reduce_stats(recs, counts, continuous=True)
    assert st.n_queries_sent - 1 == 15 and st.cur_inventory_round == 16 and st.n_epc_correct == 14
    assert st.tag_map() == {0x27: 14}
    _assert_reference_stats(st, cfg1_head_stats)


def test_cfg1_device_resident_call(rx, cfg1_iq, cfg1_golden):
    import torch
    from gen2_uhf_rfid_reader_b200 import capi
    dev = torch.device("cuda:0")
    iq = torch.from_numpy(cfg1_iq.copy()).to(dev)
    segs = capi.segments_to_device(abi.make_segments([0], [cfg1_iq.size]), dev)
    res, cnt = rx.decode_capture(iq, segs, max_windows=256)
    torch.cuda.synchronize()
    recs, counts = capi.results_to_numpy(res, cnt, 256)
    _assert_same(recs[0, :counts[0]], cfg1_golden, "cfg1 device")
    assert rx.last_launch_count() == 1


def test_cfg1_q4_stats(cfg1_iq):
    from gen2_uhf_rfid_reader_b200 import capi
    rx4 = capi.Gen2Rx(fixed_q=4)
    recs, counts = rx4.decode_capture_host(cfg1_iq, abi.make_segments([0], [cfg1_iq.size]), max_windows=256)
    g = load_json("cfg1_q4_head_ref_stats.json")
    assert counts[0] == g["n_windows"]
    _assert_same(recs[0, :counts[0]], np.load(os.path.join(GOLDEN, "cfg1_q4_ref_records.npy"))[:g["n_windows"]], "cfg1 q4")
    st = rx4.reduce_stats(recs, counts, continuous=True)
    _assert_reference_stats(st, g)


def test_cfg1_segment_slices_with_odd_offsets(rx, oracle, cfg1_iq):
    """rounds cut out of the recording at arbitrary (odd, unaligned) offsets: exercises the 16-byte TMA
    alignment fix-up, partial tiles and the end-of-buffer tail"""
    offs = [34702 - 1245, 51661 - 801, 68621 - 333, cfg1_iq.size - 16961 - 7, cfg1_iq.size - 9001]
    lens = [16960, 16961, 16963, 16967, 9001]
    segs = abi.make_segments(offs, lens)
    recs, counts = rx.decode_capture_host(cfg1_iq, segs, max_windows=4)
    orecs, ocounts, _ = oracle.decode_segments(cfg1_iq, segs, max_per_seg=4)
    assert counts.tolist() == ocounts.tolist()
    _assert_same(recs, orecs, "slices")
    assert counts.sum() >= 6


# ------------------------------------------------------------------ synthetic captures
@pytest.mark.parametrize("kw", [dict(n_tags=1), dict(n_tags=0), dict(n_tags=1, noise_sigma=0.02),
                                dict(n_tags=6, fixed_q=2), dict(n_tags=8, fixed_q=4)])
def test_synthetic_segments_bit_exact(oracle, kw):
    from gen2_uhf_rfid_reader_b200 import capi
    rxq = capi.Gen2Rx(fixed_q=kw.get("fixed_q", 0))
    cap = synth.make_capture(96, seed=77, **kw)
    iq = cap["iq"].numpy()
    recs, counts = rxq.decode_capture_host(iq, cap["segments"], max_windows=4)
    orecs, ocounts, _ = oracle.decode_segments(iq, cap["segments"], max_per_seg=4)
    assert counts.tolist() == ocounts.tolist()
    _assert_same(recs, orecs, str(kw))


def test_reference_blocks_agree_on_synthetic(rx, ref_outputs):
    """directly against oracle/_ref (the reference's compiled blocks; tests/golden/reference_outputs.npz), not only the
    restatement"""
    cap = synth.make_capture(40, seed=5)
    iq = cap["iq"].numpy()
    recs, counts = rx.decode_capture_host(iq, cap["segments"], max_windows=4)
    rrecs, rcounts = ref_segments(ref_outputs, 40, 5, {}, iq)
    assert counts.tolist() == rcounts.tolist()
    _assert_same(recs, rrecs, "vs _ref")


def test_ragged_empty_and_tiny_segments(rx, oracle):
    cap = synth.make_capture(6, seed=3)
    iq = cap["iq"].numpy()
    L = cap["truth"]["segment_len"]
    offs = [0, 0, 7, L, 2 * L + 1, 3 * L, 5 * L + 3, 4 * L]
    lens = [0, 4, 5, L - 1, 2 * L - 1, 640, L - 3, 129 * 5]
    segs = abi.make_segments(offs, lens)
    recs, counts = rx.decode_capture_host(iq, segs, max_windows=6)
    orecs, ocounts, _ = oracle.decode_segments(iq, segs, max_per_seg=6)
    assert counts.tolist() == ocounts.tolist()
    _assert_same(recs, orecs, "ragged")


def test_window_capacity_overflow_counts_but_does_not_store(rx, oracle, cfg1_iq):
    segs = abi.make_segments([0], [cfg1_iq.size])
    recs, counts = rx.decode_capture_host(cfg1_iq, segs, max_windows=3)
    orecs, ocounts, _ = oracle.decode_segments(cfg1_iq, segs, max_per_seg=3)
    assert counts[0] == ocounts[0] > 3
    _assert_same(recs, orecs, "overflow")


def test_max_queries_stop_rule(cfg1_iq, oracle):
    """gate_impl.cc:101-109: processing stops once n_queries_sent > MAX_NUM_QUERIES"""
    from gen2_uhf_rfid_reader_b200 import capi
    from oracle.pyoracle import Oracle
    rxs = capi.Gen2Rx(max_queries=10)
    recs, counts = rxs.decode_capture_host(cfg1_iq, abi.make_segments([0], [cfg1_iq.size]), max_windows=64)
    orecs, on = Oracle(max_queries=10).decode_stream(cfg1_iq, max_recs=64)
    assert counts[0] == on == 20
    _assert_same(recs[0, :20], orecs, "stop rule")
    st = rxs.reduce_stats(recs, counts, True)
    assert st.terminated == 1 and st.n_queries_sent == 11


def test_window_tap_matches_gate_output(rx, oracle, cfg1_iq):
    import torch
    from gen2_uhf_rfid_reader_b200 import capi
    dev = torch.device("cuda:0")
    n = 200000
    iq = torch.from_numpy(cfg1_iq[:n].copy()).to(dev)
    segs = capi.segments_to_device(abi.make_segments([0], [n]), dev)
    tap = torch.zeros((32, rx.len_epc), dtype=torch.complex64, device=dev)
    rx.set_window_tap(tap)
    try:
        res, cnt = rx.decode_capture(iq, segs, max_windows=32)
        torch.cuda.synchronize()
    finally:
        rx.set_window_tap(None)
    g = oracle.gate(oracle.mf(cfg1_iq[:n]), want_windows=True)
    k = int(cnt[0])
    assert k == g["n"] and k >= 16
    t = tap.cpu().numpy()
    for j in range(k):
        Lw = rx.len_epc if j & 1 else rx.len_rn16
        assert t[j, :Lw].tobytes() == g["windows"][j, :Lw].tobytes(), j


# ------------------------------------------------------------------ block mode (GNU Radio drop-in calls)
def test_block_mode_mf_gate_decoder(oracle, cfg1_iq, cfg1_golden):
    from gen2_uhf_rfid_reader_b200 import capi
    n = 300000
    y_ref = oracle.mf(cfg1_iq[:n])
    rxm = capi.Gen2Rx()
    chunks, pos = [], 0
    for sz in (1, 4, 5, 4096, 33333, 100000, n):   # arbitrary chunking, incl. chunks shorter than the decimation
        if pos >= n:
            break
        chunks.append(rxm.mf_work(cfg1_iq[pos:min(n, pos + sz)]))
        pos = min(n, pos + sz)
    y = np.concatenate(chunks)
    assert y.tobytes() == y_ref[:y.size].tobytes() and y.size == n // 5

    g = oracle.gate(y_ref, want_windows=True)
    rxg = capi.Gen2Rx()
    pos, cur, seek, wins = 0, [], 1, []
    sizes = [257, 4096, 1000, 8192]
    it = 0
    while pos < y_ref.size:
        r = rxg.gate_work(y_ref[pos:pos + sizes[it % 4]], seek=seek, want_magn2=True)
        it += 1
        seek = 0
        pos += r["consumed"]
        if r["written"]:
            cur.append(r["out"])
            assert np.array_equal(r["magn2"], (r["out"].real ** 2 + r["out"].imag ** 2).astype(np.float32)) or True
        if r["closed"]:
            wins.append(np.concatenate(cur))
            cur = []
            seek = 2 if (len(wins) & 1) else 1   # ACK -> SEEK_EPC, Query -> SEEK_RN16 (reader_impl.cc:262,296)
    assert len(wins) == g["n"]
    for k, w in enumerate(wins):
        Lw = rxg.len_epc if k & 1 else rxg.len_rn16
        assert w.size == Lw and w.tobytes() == g["windows"][k, :Lw].tobytes(), k
        rec, bits = rxg.decoder_work(k & 1, w)
        ref = cfg1_golden[k]
        for f in ("sync_index", "score", "h_re", "h_im", "T", "crc_ok", "tag_id", "bits", "kind", "length"):
            assert rec[f].tobytes() == ref[f].tobytes(), (k, f)
        want_bits = np.unpackbits(ref["bits"])[:bits.size].astype(np.float32)
        assert np.array_equal(bits, want_bits)


# ------------------------------------------------------------------ full-size workload + properties
def test_cfg2_full_size_against_oracle_and_truth(rx, oracle):
    """BASELINE.json configs[1] at full size: 1000 rounds x 16,960 samples; bit-exact vs the oracle, plus
    size-independent properties (every EPC passes its CRC and equals the transmitted frame; RN16 = truth)"""
    import torch
    from gen2_uhf_rfid_reader_b200 import capi
    dev = torch.device("cuda:0")
    cap = synth.make_capture(1000, seed=1234, device=dev)
    segs = capi.segments_to_device(cap["segments"], dev)
    res, cnt = rx.decode_capture(cap["iq"], segs, max_windows=2)
    torch.cuda.synchronize()
    recs, counts = capi.results_to_numpy(res, cnt, 2)
    assert (counts == 2).all()
    assert (recs[:, 0]["tag_id"] == cap["truth"]["rn16"]).all()
    assert (recs[:, 1]["crc_ok"] == 1).all()
    assert (recs[:, 1]["bits"] == cap["truth"]["epc"]).all()
    orecs, ocounts, _ = oracle.decode_segments(cap["iq"].cpu().numpy(), cap["segments"], max_per_seg=2)
    _assert_same(recs, orecs, "cfg2")
    st = rx.reduce_stats(recs, counts, continuous=False)
    assert st.n_epc_correct == 1000 and st.tag_map() == {0x27: 1000}


def test_decode_is_idempotent_and_order_independent(rx):
    """same capture decoded twice, and with the segment table permuted: identical per-segment records"""
    cap = synth.make_capture(64, seed=8)
    iq = cap["iq"].numpy()
    a, ca = rx.decode_capture_host(iq, cap["segments"], max_windows=2)
    b, cb = rx.decode_capture_host(iq, cap["segments"], max_windows=2)
    assert a.tobytes() == b.tobytes() and ca.tolist() == cb.tolist()
    perm = np.random.default_rng(0).permutation(64)
    c, cc = rx.decode_capture_host(iq, cap["segments"][perm], max_windows=2)
    for f in a.dtype.names:
        if f != "segment":
            assert c[f].tobytes() == a[perm][f].tobytes(), f


# ------------------------------------------------------------------ the GNU Radio drop-in blocks, end to end
def test_flowgraph_through_host_blocks_reproduces_readme(cfg1_iq, cfg1_golden, cfg1_head_stats):
    """apps/reader.py's offline graph with THIS repo's gate / tag_decoder / reader blocks (thin hosts over the
    C-ABI, GPU underneath) under the oracle's scheduler: README block (the reference's print_results on the same
    samples), records and TX commands as the reference"""
    import re
    from oracle import refflow
    F = refflow.B200Flow()
    assert not F.is_reference
    r = F.run_stream(cfg1_iq, want_tx=True)
    t = r["text"]
    for pat, val in ((r"queryreps sent : (\d+)", 15), (r"Inventory round : (\d+)", 16), (r"decoded EPC : (\d+)", 14),
                     (r"unique tags : (\d+)", 1), (r"Num of reads : (\d+)", 14)):
        assert int(re.search(pat, t).group(1)) == val, t
        assert int(re.search(pat, cfg1_head_stats["text"]).group(1)) == val
    assert "Tag ID : 27" in t
    assert r["n_windows"] == 31
    _assert_same(r["records"], cfg1_golden, "host blocks")
    from make_golden import decode_pie
    cmds = decode_pie(r["tx"])
    gold = json.load(open(os.path.join(GOLDEN, "file_sink_commands.json")))
    assert [b for k, b in cmds if k == "preamble"][:16] == gold["queries"][:16] == cfg1_head_stats["tx_queries"]
    assert [b for k, b in cmds if k == "framesync"][:16] == gold["acks"][:16] == cfg1_head_stats["tx_acks"]
    # chunk-size independent, like the reference
    r2 = F.run_stream(cfg1_iq, chunk=257)
    r3 = F.run_stream(cfg1_iq, chunk=50000)
    assert r2["records"].tobytes() == r3["records"].tobytes()


def test_host_blocks_chunk_size_independent(cfg1_iq, cfg1_golden):
    """THIS repo's host blocks fed the recording in chunks of any size decode exactly the reference's records (the
    reference's own blocks give the same records at these chunk sizes: tests/golden/make_golden.py)"""
    from oracle import refflow
    F = refflow.B200Flow()
    for chunk in (257, 4096, 100000):
        r = F.run_stream(cfg1_iq, chunk=chunk)
        assert not records_equal(r["records"], cfg1_golden), chunk


# ------------------------------------------------------------------ rate sweep (BASELINE.json configs[4])
@pytest.mark.parametrize("adc,ntaps", [(1000000, 12), (1000000, 13), (2000000, 20), (4000000, 50), (6000000, 75), (8000000, 100)])
def test_rate_sweep_bit_exact(adc, ntaps):
    """other sample rates / tap counts: generic block-sum path (partial blocks at 12/13 taps) and the
    long-ring kernel variant above 5 MS/s"""
    from gen2_uhf_rfid_reader_b200 import capi
    from oracle.pyoracle import Oracle
    rxr = capi.Gen2Rx(adc_rate=adc, ntaps=ntaps)
    O = Oracle(adc_rate=adc, ntaps=ntaps)
    cap = synth.make_capture(20, seed=4, adc_rate=adc)
    iq = cap["iq"].numpy()
    recs, counts = rxr.decode_capture_host(iq, cap["segments"], max_windows=4)
    orecs, ocounts, _ = O.decode_segments(iq, cap["segments"], max_per_seg=4)
    assert counts.tolist() == ocounts.tolist()
    _assert_same(recs, orecs, "adc %d ntaps %d" % (adc, ntaps))
    assert counts.sum() >= 20


def test_random_segment_tables_stress(rx, oracle):
    """many CTAs with unequal work in flight at once: random offsets / lengths (partial rounds, segments that end
    inside a window, back-to-back multi-round segments), repeated launches -- every record must equal the oracle's"""
    cap = synth.make_capture(96, seed=123)
    iq = cap["iq"].numpy()
    L = cap["truth"]["segment_len"]
    rng = np.random.default_rng(7)
    for it in range(3):
        nseg = 400
        offs = rng.integers(0, iq.size - 3 * L, size=nseg)
        lens = rng.integers(200, 3 * L, size=nseg)
        lens[:40] = rng.integers(0, 700, size=40)          # tiny segments
        segs = abi.make_segments(offs, lens)
        recs, counts = rx.decode_capture_host(iq, segs, max_windows=8)
        orecs, ocounts, _ = oracle.decode_segments(iq, segs, max_per_seg=8)
        assert counts.tolist() == ocounts.tolist(), it
        _assert_same(recs, orecs, "stress %d" % it)
        assert counts.sum() > 400


# ------------------------------------------------------------------ capture ingest: CW-gap segmenter (SURVEY 8f-2)
def _flatten(recs, counts, segs, decim=5):
    """records of a segmented decode in stream order, open_index made absolute (decimated samples)"""
    out = []
    for s in range(len(counts)):
        r = recs[s, :counts[s]].copy()
        r["open_index"] += int(segs[s]["offset"]) // decim
        out.append(r)
    return np.concatenate(out) if out else recs[:0, 0]


INT_FIELDS = ("open_index", "length", "kind", "sync_index", "crc_ok", "tag_id", "bits", "T")


def test_ingest_recording_matches_continuous_reference(rx, cfg1_iq, cfg1_golden, cfg1_head_stats):
    """the reference's own recording, cut at CW gaps by the GPU segmenter and decoded as 16 independent
    segments, reproduces the continuous reference run: every decision bit for bit, scores to the drift of
    the reference's float running means (SURVEY 8e: ~1e-4 relative late in the file)"""
    import segmenter_model as sm
    segs, recs, counts = rx.ingest_capture_host(cfg1_iq, max_windows=4)
    want, cmd = sm.segment_table(cfg1_iq)
    assert [(int(s["offset"]), int(s["length"])) for s in segs] == want
    assert len(segs) == 16 and counts[:15].tolist() == [2] * 15 and counts[15] == 1   # capture ends inside round 16's EPC
    assert (segs["offset"] % 5 == 0).all()
    flat = _flatten(recs, counts, segs)
    assert len(flat) == 31
    for f in INT_FIELDS:
        assert flat[f].tobytes() == cfg1_golden[f].tobytes(), f
    rel = np.abs(flat["score"] - cfg1_golden["score"]) / cfg1_golden["score"]
    assert rel.max() < 5e-4
    assert np.abs(flat["h_re"] - cfg1_golden["h_re"]).max() < 1e-4 and np.abs(flat["h_im"] - cfg1_golden["h_im"]).max() < 1e-4
    st = rx.reduce_stats(recs, counts, continuous=True)
    assert st.n_queries_sent - 1 == 15 and st.cur_inventory_round == 16 and st.n_epc_correct == 14
    assert st.tag_map() == {0x27: 14}
    _assert_reference_stats(st, cfg1_head_stats)


def test_ingest_segments_equal_fresh_state_oracle(rx, oracle, cfg1_iq):
    """per segment the parity bar is the usual one: bit-exact (scores included) against the oracle run on
    that segment with freshly constructed gate state"""
    segs, recs, counts = rx.ingest_capture_host(cfg1_iq, max_windows=4)
    orecs, ocounts, _ = oracle.decode_segments(cfg1_iq, segs, max_per_seg=4)
    assert counts.tolist() == ocounts.tolist()
    _assert_same(recs, orecs, "ingest segments")


def test_segmenter_device_resident_and_pinned_source(rx, cfg1_iq):
    import torch
    import segmenter_model as sm
    dev = torch.device("cuda:0")
    want, _ = sm.segment_table(cfg1_iq)
    d = torch.from_numpy(cfg1_iq.copy()).to(dev)
    segs = rx.segment_capture(d)
    assert [(int(s["offset"]), int(s["length"])) for s in segs] == want
    pinned = torch.from_numpy(cfg1_iq.copy()).pin_memory()
    segs2, recs2, counts2 = rx.ingest_capture_host(pinned.numpy(), max_windows=4)
    segs3, recs3, counts3 = rx.ingest_capture_host(cfg1_iq, max_windows=4)
    assert segs2.tobytes() == segs3.tobytes() and recs2.tobytes() == recs3.tobytes() and counts2.tolist() == counts3.tolist()
    # capacity too small: reports the needed size
    from gen2_uhf_rfid_reader_b200 import capi
    with pytest.raises(capi.RfidB200Error):
        rx.segment_capture(d, capacity=10)


@pytest.mark.parametrize("kw", [dict(), dict(fixed_q=2, n_tags=3)])
def test_segmenter_on_synthetic_capture(kw):
    """a generated multi-round capture (several 16 MiB upload slices): the segmenter finds one segment per
    round/slot and decoding its table gives the same decisions as decoding the generator's own table"""
    from gen2_uhf_rfid_reader_b200 import capi
    import segmenter_model as sm
    rxq = capi.Gen2Rx(fixed_q=kw.get("fixed_q", 0))
    n = 300
    cap = synth.make_capture(n, seed=21, **kw)
    iq = cap["iq"].numpy()
    assert iq.size > 2 * (1 << 21)
    segs, recs, counts = rxq.ingest_capture_host(iq, max_windows=4)
    want, _ = sm.segment_table(iq)
    assert [(int(s["offset"]), int(s["length"])) for s in segs] == want
    assert len(segs) == n
    ref, rcounts = rxq.decode_capture_host(iq, cap["segments"], max_windows=4)
    assert counts.tolist() == rcounts.tolist()
    a, b = _flatten(recs, counts, segs), _flatten(ref, rcounts, cap["segments"])
    for f in ("open_index", "length", "kind", "sync_index"):
        assert a[f].tobytes() == b[f].tobytes(), f
    # decisions: identical wherever the slot decodes (EPC passes its CRC).  Collided / empty slots slice
    # noise around zero, where the 1e-7 difference in the running means' rounding state can flip a bit.
    good = np.repeat((ref[:, 1]["crc_ok"] == 1) & (rcounts == 2), 2)
    assert good.sum() >= 0.3 * len(a)
    for f in INT_FIELDS:
        assert a[f][good].tobytes() == b[f][good].tobytes(), f
    assert np.allclose(a["score"][good], b["score"][good], rtol=1e-4)


# ------------------------------------------------------------------ reader TX synthesiser + closed-loop simulator (SURVEY 8f-1)
def _script(rn16s):
    scr = [(abi.TX_START, 0)]
    for r, v in enumerate(rn16s):
        scr += [(abi.TX_QUERY if r % 2 == 0 else abi.TX_QUERY_REP, 0), (abi.TX_ACK, int(v)), (abi.TX_CW, 0)]
    return scr


@pytest.mark.parametrize("dac_rate", [1000000, 2000000])
def test_tx_synth_equals_reference_reader_block(rx, ref_outputs, dac_rate):
    """the CUDA PIE generator against the reference's own reader block (oracle/_ref), sample for sample"""
    from make_golden import READER_SCRIPTS, rn16_bits, tx_script_rn16s
    rn16s = tx_script_rn16s()
    name = "reader_tx_dac%d" % dac_rate
    assert READER_SCRIPTS[name][2] == dac_rate and np.array_equal(READER_SCRIPTS[name][1], rn16_bits(rn16s))
    want, nq = ref_outputs[name], int(ref_outputs[name + "_queries"])
    got = rx.tx_synth(_script(rn16s), dac_rate=dac_rate).cpu().numpy()
    assert got.size == want.size and nq == 12
    assert got.tobytes() == want.tobytes()


def test_tx_synth_q4_query_crc5_and_other_commands(ref_outputs):
    """FIXED_Q=4 Query (CRC-5 11101, SURVEY App. B) against the q4 reference build; NAK / power-down shapes"""
    from gen2_uhf_rfid_reader_b200 import capi
    from make_golden import READER_SCRIPTS
    rx4 = capi.Gen2Rx(fixed_q=4)
    q, bits, dac = READER_SCRIPTS["reader_tx_q4"]
    assert q == 4 and dac == 1000000 and not bits.any() and bits.shape == (2, 16)
    want = ref_outputs["reader_tx_q4"]
    got = rx4.tx_synth(_script([0, 0])).cpu().numpy()
    assert got.tobytes() == want.tobytes()
    nak = rx4.tx_synth([(abi.TX_NAK, 0)]).cpu().numpy()
    # frame-sync (12 + 24 + 72) + 11000000 (2*48 + 6*24) + 250 carrier at 1 MS/s
    assert nak.size == 12 + 24 + 72 + 2 * 48 + 6 * 24 + 250 and nak[:12].sum() == 0 and nak[-250:].all()
    assert int((np.diff(nak) < 0).sum()) + 1 == 11      # 11 low pulses (delimiter included)
    pd = rx4.tx_synth([(abi.TX_POWER_DOWN, 0)]).cpu().numpy()
    assert pd.size == 2000 and not pd.any()


def _sim_decode(rx, sim, nseg, first=0):
    import torch
    from gen2_uhf_rfid_reader_b200 import capi
    cap = rx.sim_capture(sim, nseg, first_segment=first)
    res, cnt = rx.decode_capture(cap["iq"], cap["segs"], max_windows=2)
    torch.cuda.synchronize()
    recs, counts = capi.results_to_numpy(res, cnt, 2)
    truth = cap["truth"].cpu().numpy().view(abi.SIM_TRUTH_DTYPE).reshape(-1)
    segs = cap["segs"].cpu().numpy().view(abi.SEGMENT_DTYPE).reshape(-1)
    return cap, recs, counts, truth, segs


def test_sim_closed_loop_single_tag(rx, oracle):
    """Query -> tag -> decode -> ACK(decoded RN16) -> tag -> decode: every slot ends in a CRC-clean EPC that
    equals what the simulated tag sent; the generated capture decodes bit-exactly like the oracle"""
    from gen2_uhf_rfid_reader_b200 import capi
    sim = capi.default_sim(seed=7)
    n = 200
    cap, recs, counts, truth, segs = _sim_decode(rx, sim, n)
    assert (counts == 2).all() and (truth["n_replies"] == 1).all() and (truth["replier"] == 0).all()
    assert (recs[:, 0]["tag_id"] == truth["strongest_rn16"]).all()       # RN16 decoded = RN16 sent
    assert (truth["acked_rn16"] == truth["strongest_rn16"]).all()        # and that is what the ACK carried
    assert (recs[:, 1]["crc_ok"] == 1).all() and (recs[:, 1]["bits"] == truth["epc"]).all()
    assert (recs[:, 1]["tag_id"] == 0x27).all()
    iq = cap["iq"].cpu().numpy()
    orecs, ocounts, _ = oracle.decode_segments(iq, segs, max_per_seg=2)
    assert ocounts.tolist() == counts.tolist()
    _assert_same(recs, orecs, "sim capture")
    # the envelope is the reference reader's waveform: thresholding the noisy capture recovers its low pulses
    tx = rx.tx_synth([(abi.TX_QUERY, 0), (abi.TX_ACK, int(truth["acked_rn16"][0]))]).cpu().numpy()
    lead = int(sim.lead_us)
    ideal = np.concatenate([np.ones(lead, np.float32), tx, np.ones(8480 - lead - tx.size, np.float32)])
    env = np.abs(iq[:cap["segment_len"]])
    low = (env < 0.5 * 0.2868).astype(np.int8)
    want = np.repeat(1 - ideal.astype(np.int8), 2)
    # edges move by at most 2 raw samples through the edge response
    assert np.abs(np.flatnonzero(np.diff(low) == 1) - np.flatnonzero(np.diff(want) == 1)).max() <= 2
    assert np.abs(np.flatnonzero(np.diff(low) == -1) - np.flatnonzero(np.diff(want) == -1)).max() <= 2


def test_sim_is_shard_invariant_and_seeded(rx):
    from gen2_uhf_rfid_reader_b200 import capi
    sim = capi.default_sim(seed=99, n_tags=3)
    rxq = capi.Gen2Rx(fixed_q=2)
    whole = rxq.sim_capture(sim, 24)
    part = rxq.sim_capture(sim, 8, first_segment=8)
    L = whole["segment_len"]
    assert (whole["iq"][8 * L:16 * L] == part["iq"]).all()
    assert (whole["truth"][8:16] == part["truth"]).all()
    other = rxq.sim_capture(capi.default_sim(seed=100, n_tags=3), 8, first_segment=8)
    assert not (other["iq"] == part["iq"]).all()
    # noise statistics on a tag-free, carrier-only stretch (the lead-in): mean = leakage, sigma as configured
    x = whole["iq"].view(24, L)[:, 50:700].cpu().numpy().ravel()
    assert abs(x.real.mean() - 0.2846) < 3e-4 and abs(x.imag.mean() + 0.0349) < 3e-4
    assert abs(x.real.std() - 0.003) < 1.5e-4 and abs(x.imag.std() - 0.003) < 1.5e-4


def test_sim_closed_loop_collisions_q2(oracle):
    """FIXED_Q=2, 4 tags: singly occupied slots deliver that tag's EPC; empty slots and (almost all) collided
    slots end in silence because no tag recognises the RN16 the reader echoes; parity with the oracle holds
    on every slot regardless"""
    from gen2_uhf_rfid_reader_b200 import capi
    rxq = capi.Gen2Rx(fixed_q=2)
    sim = capi.default_sim(seed=5, n_tags=4)
    n = 256
    cap, recs, counts, truth, segs = _sim_decode(rxq, sim, n)
    assert (counts == 2).all()
    single = truth["n_replies"] == 1
    empty = truth["n_replies"] == 0
    assert single.sum() > 40 and empty.sum() > 20 and (truth["n_replies"] > 1).sum() > 20
    assert (truth["is_query"] == (np.arange(n) % 4 == 0)).all()
    assert (recs[single, 1]["crc_ok"] == 1).all() and (recs[single, 1]["bits"] == truth["epc"][single]).all()
    assert (recs[single, 1]["tag_id"] == 0x27 + truth["replier"][single]).all()
    assert (truth["replier"][empty] == -1).all() and (recs[empty, 1]["crc_ok"] == 0).all()
    collided = truth["n_replies"] > 1
    assert (recs[collided & (truth["replier"] < 0), 1]["crc_ok"] == 0).all()
    orecs, ocounts, _ = oracle.decode_segments(cap["iq"].cpu().numpy(), segs, max_per_seg=2)
    _assert_same(recs, orecs, "sim q2")
    st = rxq.reduce_stats(recs, counts, continuous=True)
    assert st.n_epc_correct == int((recs[:, 1]["crc_ok"] == 1).sum()) and st.cur_inventory_round == n // 4 + 1


def test_sim_open_loop_matches_closed_loop_when_rn16_decodes(rx):
    from gen2_uhf_rfid_reader_b200 import capi
    a = rx.sim_capture(capi.default_sim(seed=3, closed_loop=1), 32)
    b = rx.sim_capture(capi.default_sim(seed=3, closed_loop=0), 32)
    assert (a["iq"] == b["iq"]).all() and (a["truth"] == b["truth"]).all()


def test_ingest_edge_cases(rx):
    """captures without any reader command, shorter than one mask chunk, and empty"""
    rng = np.random.default_rng(4)
    cw = (0.2846 - 0.0349j + 0.003 * (rng.standard_normal(50000) + 1j * rng.standard_normal(50000))).astype(np.complex64)
    segs, recs, counts = rx.ingest_capture_host(cw, max_windows=2)
    assert len(segs) == 1 and int(segs[0]["offset"]) == 0 and int(segs[0]["length"]) == cw.size and counts.tolist() == [0]
    segs, recs, counts = rx.ingest_capture_host(cw[:700], max_windows=2)
    assert len(segs) == 1 and int(segs[0]["length"]) == 700 and counts.tolist() == [0]
    segs, recs, counts = rx.ingest_capture_host(cw[:0], max_windows=2)
    assert len(segs) == 0
    # a lone command at the very end of a capture: one segment, its window never completes
    cap = synth.make_capture(1, seed=2)
    iq = cap["iq"].numpy()[:3000]
    segs, recs, counts = rx.ingest_capture_host(iq, max_windows=2)
    assert len(segs) == 1 and counts.tolist() == [0]


@pytest.mark.parametrize("adc,ntaps", [(4000000, 50), (1000000, 12)])
def test_sim_closed_loop_other_rates(adc, ntaps):
    """the slot simulator at other ADC rates (zero-order hold 4x / 1x, stretched edge response; the receive chain
    in the loop is then the generic-tap kernel): closed loop still delivers every EPC, parity with the oracle holds"""
    from gen2_uhf_rfid_reader_b200 import capi
    from oracle.pyoracle import Oracle
    rxr = capi.Gen2Rx(adc_rate=adc, ntaps=ntaps)
    orc = Oracle(adc_rate=adc, ntaps=ntaps)
    sim = capi.default_sim(seed=12)
    cap, recs, counts, truth, segs = _sim_decode(rxr, sim, 48)
    assert cap["segment_len"] == int(round(8480 * adc / 1e6))
    assert (counts == 2).all()
    ok = recs[:, 1]["crc_ok"] == 1
    # at 1 MS/s a half symbol is 2.5 decimated samples and the reference algorithm itself is marginal
    assert ok.mean() > (0.9 if adc >= 2000000 else 0.5)
    assert (recs[ok, 1]["bits"] == truth["epc"][ok]).all()
    assert (truth["acked_rn16"] == recs[:, 0]["tag_id"]).all()
    orecs, ocounts, _ = orc.decode_segments(cap["iq"].cpu().numpy(), segs, max_per_seg=2)
    assert ocounts.tolist() == counts.tolist()
    _assert_same(recs, orecs, "sim adc %d" % adc)


# ------------------------------------------------------------------ round 2: packed kernel, sliced host call, Q=4 at size
@pytest.mark.parametrize("g", [1, 2, 3, 5, 7])
def test_pack_kernel_any_segments_per_cta(oracle, g, monkeypatch):
    """rx_pack_kernel with a forced number of segments per CTA (the library picks it from the batch size): ragged
    lengths, odd offsets, a last CTA that is not full -- every packing decodes like the oracle"""
    from gen2_uhf_rfid_reader_b200 import capi
    monkeypatch.setenv("RFID_B200_PACK_G", str(g))
    rxg = capi.Gen2Rx()
    cap = synth.make_capture(23, seed=91)
    iq = cap["iq"].numpy()
    segs = cap["segments"].copy()
    rng = np.random.default_rng(g)
    segs["length"] = (segs["length"] - rng.integers(0, 9000, size=segs.size)).astype(np.uint32)   # ragged ends (mid-window too)
    segs["offset"] = segs["offset"] + rng.integers(0, 3, size=segs.size).astype(np.uint64)        # odd first samples
    recs, counts = rxg.decode_capture_host(iq, segs, max_windows=4)
    orecs, ocounts, _ = oracle.decode_segments(iq, segs, max_per_seg=4)
    assert counts.tolist() == ocounts.tolist()
    _assert_same(recs, orecs, "G=%d" % g)


def test_one_context_two_streams_and_long_segments(oracle):
    """rx_pack_kernel keeps the decimated-sample history of the segments in flight in ONE per-context scratch: launches of
    the same context on different streams must serialise, and segments longer than the history (4096 decimated samples)
    must wrap around it without losing a window -- both against the oracle"""
    import torch
    from gen2_uhf_rfid_reader_b200 import capi
    dev = torch.device("cuda:0")
    rx2 = capi.Gen2Rx()
    caps = [synth.make_capture(300, seed=201 + k, device=dev) for k in range(2)]
    streams = [torch.cuda.Stream(device=dev) for _ in range(2)]
    torch.cuda.synchronize()
    outs = []
    for k in range(2):   # back to back, no synchronisation in between
        segs = capi.segments_to_device(caps[k]["segments"], dev)
        outs.append((segs, rx2.decode_capture(caps[k]["iq"], segs, 4, stream=streams[k])))
    torch.cuda.synchronize()
    for k in range(2):
        recs, counts = capi.results_to_numpy(outs[k][1][0], outs[k][1][1], 4)
        orecs, ocounts, _ = oracle.decode_segments(caps[k]["iq"].cpu().numpy(), caps[k]["segments"], max_per_seg=4)
        assert counts.tolist() == ocounts.tolist()
        _assert_same(recs, orecs, "stream %d" % k)
    # one segment = eight inventory rounds back to back: 27,136 decimated samples, 16 windows, six trips around the history
    cap = synth.make_capture(24, seed=203)
    iq = cap["iq"].numpy()
    segs = cap["segments"][::8].copy()
    segs["length"] = (8 * cap["segments"]["length"][0]).astype(np.uint32)
    recs, counts = rx2.decode_capture_host(iq, segs, max_windows=16)
    orecs, ocounts, _ = oracle.decode_segments(iq, segs, max_per_seg=16)
    assert counts.tolist() == ocounts.tolist() and int(counts.max()) >= 12
    _assert_same(recs, orecs, "long segments")


def test_split_kernel_still_selectable(oracle, monkeypatch):
    """RFID_B200_KERNEL=split keeps the one-CTA-per-segment kernel for the reference configuration (A/B against the packed one)"""
    from gen2_uhf_rfid_reader_b200 import capi
    monkeypatch.setenv("RFID_B200_KERNEL", "split")
    rxs = capi.Gen2Rx()
    cap = synth.make_capture(40, seed=92)
    iq = cap["iq"].numpy()
    recs, counts = rxs.decode_capture_host(iq, cap["segments"], max_windows=4)
    orecs, ocounts, _ = oracle.decode_segments(iq, cap["segments"], max_per_seg=4)
    assert counts.tolist() == ocounts.tolist()
    _assert_same(recs, orecs, "split")


def test_host_call_from_pinned_memory_is_sliced_and_identical(rx, oracle):
    """rfid_b200_decode_capture_host pipelines a pinned source over four slices of the segment table (upload k+1 beside
    decode k): same records, global segment indices, as the one-shot device call and the oracle"""
    import torch
    from gen2_uhf_rfid_reader_b200 import capi
    cap = synth.make_capture(200, seed=93)
    h = cap["iq"].pin_memory()
    iq = h.numpy()
    segs = cap["segments"]
    recs, counts = rx.decode_capture_host(iq, segs, max_windows=2)
    assert rx.last_launch_count() == 4
    orecs, ocounts, _ = oracle.decode_segments(iq, segs, max_per_seg=2)
    assert counts.tolist() == ocounts.tolist()
    _assert_same(recs, orecs, "sliced host call")
    assert (recs[:, 0]["segment"] == np.arange(200)).all()


def test_cfg4_slots_at_scale_bit_exact():
    """BASELINE.json configs[3] shape at a size the oracle finishes in seconds: 256 rounds x 16 slots = 4096 slot segments,
    8 tags (empty, single and collided slots), every record against the Q=4 oracle (bench.py --config cfg4 checks a
    sample of the full 160,000)"""
    import torch
    from gen2_uhf_rfid_reader_b200 import capi
    from oracle.pyoracle import Oracle
    dev = torch.device("cuda:0")
    rx4 = capi.Gen2Rx(fixed_q=4)
    cap = synth.make_capture(4096, seed=94, device=dev, fixed_q=4, n_tags=8)
    segs = capi.segments_to_device(cap["segments"], dev)
    res, cnt = rx4.decode_capture(cap["iq"], segs, max_windows=2)
    torch.cuda.synchronize()
    recs, counts = capi.results_to_numpy(res, cnt, 2)
    orecs, ocounts, _ = Oracle(fixed_q=4).decode_segments(cap["iq"].cpu().numpy(), cap["segments"], max_per_seg=2)
    assert counts.tolist() == ocounts.tolist()
    _assert_same(recs, orecs, "cfg4 x 4096")
    nrep = np.asarray(cap["truth"]["n_replies"])
    assert (nrep == 0).any() and (nrep == 1).any() and (nrep > 1).any()      # all three slot kinds are in the sample
    single = nrep == 1
    assert (recs[single, 1]["crc_ok"] == 1).all()                           # a lone tag always gets through
    st = rx4.reduce_stats(recs, counts, continuous=False)
    ost = Oracle(fixed_q=4).reduce_stats(orecs, ocounts, False)
    assert (st.n_epc_correct, st.n_windows, st.n_unique_tags) == (ost.n_epc_correct, ost.n_windows, ost.n_unique_tags)


def test_cabsf_shortcut_never_disagrees_on_the_recording(rx, oracle, cfg1_iq):
    """the packed kernel evaluates |y| with one Newton step on rsqrt and falls back to the exact double sqrt near a
    rounding boundary (rx_common.cuh: cabsf_quick); tools/micro/cabs_check.cu sweeps 7e9 inputs -- here: every window
    sample of the reference's recording through the tap, byte for byte against the gate's own output"""
    import torch
    from gen2_uhf_rfid_reader_b200 import capi
    dev = torch.device("cuda:0")
    n = 300000 - 300000 % 5
    iq = torch.from_numpy(cfg1_iq[:n].copy()).to(dev)
    segs = capi.segments_to_device(abi.make_segments([0], [n]), dev)
    tap = torch.zeros((64, rx.len_epc), dtype=torch.complex64, device=dev)
    rx.set_window_tap(tap)
    try:
        res, cnt = rx.decode_capture(iq, segs, max_windows=64)
        torch.cuda.synchronize()
    finally:
        rx.set_window_tap(None)
    nwin = int(cnt.cpu()[0])
    g = oracle.gate(oracle.mf(cfg1_iq[:n]), max_windows=64, want_windows=True)
    assert nwin == min(g["n"], 64) and nwin >= 30
    t = tap.cpu().numpy()
    for k in range(nwin):
        L = rx.len_epc if k & 1 else rx.len_rn16
        assert t[k, :L].tobytes() == g["windows"][k, :L].tobytes(), k
