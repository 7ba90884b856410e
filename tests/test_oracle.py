"""CPU tests: the oracle is pinned to the reference's golden vectors and to the reference's own code.

Golden material (SURVEY.md section 4 / Appendix B): README.md:46-53 expected output, the RN16s the reference
author's run decoded (recovered from misc/data/file_sink), and what oracle/_ref (the reference's own blocks) computed,
stored by tests/golden/make_golden.py.
"""
import json
import os
import re

import numpy as np
import pytest

from conftest import GOLDEN, load_json, records_equal, ref_segments
from gen2_uhf_rfid_reader_b200 import abi, synth


def _readme_numbers():
    txt = open(os.path.join(GOLDEN, "readme_expected.txt")).read()
    g = lambda pat: re.search(pat, txt).group(1)  # noqa: E731
    return {"sent": int(g(r"queryreps sent : (\d+)")), "round": int(g(r"Inventory round : (\d+)")),
            "epc": int(g(r"decoded EPC : (\d+)")), "unique": int(g(r"unique tags : (\d+)")),
            "tag": int(g(r"Tag ID : (\w+)"), 16), "reads": int(g(r"Num of reads : (\d+)"))}


def test_reference_reproduces_readme():
    """the compiled reference + our scheduler print the README block (README.md:48-53) on the whole recording
    (the run's print_results text is stored in cfg1_ref_stats.json)"""
    t = load_json("cfg1_ref_stats.json")["text"]
    exp = _readme_numbers()
    assert "queryreps sent : %d" % exp["sent"] in t
    assert "Inventory round : %d" % exp["round"] in t
    assert "decoded EPC : %d" % exp["epc"] in t
    assert "unique tags : %d" % exp["unique"] in t
    assert "Tag ID : %x  Num of reads : %d" % (exp["tag"], exp["reads"]) in t
    assert exp == {"sent": 71, "round": 72, "epc": 70, "unique": 1, "tag": 0x27, "reads": 70}


def test_golden_rn16_match_author_run(cfg1_full_golden):
    """the 71 RN16s decoded on file_source_test are the ones ACKed in the author's TX file misc/data/file_sink"""
    cmds = json.load(open(os.path.join(GOLDEN, "file_sink_commands.json")))
    assert len(cmds["queries"]) == 72 and len(cmds["acks"]) == 71
    assert set(cmds["queries"]) == {"1000000000000000010000"}
    rn = [abi.bits_hex(r) for r in cfg1_full_golden if r["kind"] == abi.RN16]
    assert rn == cmds["rn16"]
    assert all(a.startswith("01") for a in cmds["acks"])


def test_reference_tx_matches_author_run(cfg1_head_stats):
    """the reader block's own TX envelope (driven by our scheduler over cfg1_iq; its commands are stored in
    cfg1_head_ref_stats.json) = the committed file_sink, command by command"""
    gold = json.load(open(os.path.join(GOLDEN, "file_sink_commands.json")))
    q, a = cfg1_head_stats["tx_queries"], cfg1_head_stats["tx_acks"]
    assert len(q) == cfg1_head_stats["n_queries_sent"] == 16 and len(a) == 16
    assert q == gold["queries"][:len(q)] and a == gold["acks"][:len(a)]


def test_restatement_equals_reference_on_cfg1(oracle, cfg1_iq, cfg1_golden):
    recs, n = oracle.decode_stream(cfg1_iq)
    assert n == 31
    assert not records_equal(recs, cfg1_golden)
    # facts recorded in SURVEY.md 8(c); the whole recording's last window opens at 246811
    assert list(recs["open_index"][:4]) == [7393, 8731, 11302, 12123] and recs["open_index"][-1] == 58751
    epc = [abi.bits_hex(r) for r in recs if r["kind"] == abi.EPC and r["crc_ok"] == 1]
    assert len(epc) == 14 and set(epc) == {"3000300833b2ddd90140000000276d3e"}
    assert recs[1]["crc_ok"] == 0  # the one failed round: late ACK


def test_stats_reduction_matches_reference(oracle, cfg1_full_golden):
    st = oracle.reduce_stats(cfg1_full_golden[None, :], np.array([len(cfg1_full_golden)]), True)
    g = json.load(open(os.path.join(GOLDEN, "cfg1_ref_stats.json")))
    assert (st.n_queries_sent, st.cur_inventory_round, st.cur_slot_number, st.n_epc_correct) == \
        (g["n_queries_sent"], g["cur_inventory_round"], g["cur_slot_number"], g["n_epc_correct"])
    assert st.tag_map() == {int(k): v for k, v in g["tag_reads"].items()}
    from oracle.pyoracle import Oracle
    q4 = np.load(os.path.join(GOLDEN, "cfg1_q4_ref_records.npy"))
    g4 = json.load(open(os.path.join(GOLDEN, "cfg1_q4_ref_stats.json")))
    st4 = Oracle(fixed_q=4).reduce_stats(q4[None, :], np.array([len(q4)]), True)
    assert (st4.n_queries_sent, st4.cur_inventory_round, st4.cur_slot_number, st4.n_epc_correct) == \
        (g4["n_queries_sent"], g4["cur_inventory_round"], g4["cur_slot_number"], g4["n_epc_correct"])


@pytest.mark.parametrize("kw", [dict(n_tags=1), dict(n_tags=0), dict(n_tags=6, fixed_q=2), dict(n_tags=1, noise_sigma=0.02)])
def test_restatement_equals_reference_on_synthetic(oracle, ref_outputs, kw):
    cap = synth.make_capture(48, seed=21, **kw)
    iq = cap["iq"].numpy()
    rr, rc = ref_segments(ref_outputs, 48, 21, kw, iq)
    orr, oc, _ = oracle.decode_segments(iq, cap["segments"], max_per_seg=4)
    assert (rc == oc).all()
    assert not records_equal(rr, orr)
    if kw.get("n_tags") == 1 and "noise_sigma" not in kw:
        assert (rr[:, 0]["tag_id"] == cap["truth"]["rn16"]).all()
        assert (rr[:, 1]["crc_ok"] == 1).all()


def test_mf_order_does_not_change_decisions(oracle, cfg1_iq):
    """matched-filter summation order is unpinned by the reference; decode results do not depend on it"""
    outs = [oracle.decode_decimated(oracle.mf(cfg1_iq, v))[0] for v in (0, 1, 2)]
    for o in outs[1:]:
        for f in ("open_index", "sync_index", "T", "crc_ok", "tag_id", "bits"):
            assert o[f].tobytes() == outs[0][f].tobytes(), f
        assert np.max(np.abs(o["score"] - outs[0]["score"]) / outs[0]["score"]) < 2e-4


def test_blocked_matched_filter_is_the_canonical_one(oracle):
    """The CPU reference arm of bench.py times the canonical boxcar with every block sum formed once (variant 3):
    it must be the canonical order bit for bit, for any length and tap count"""
    rng = np.random.default_rng(5)
    for n in (0, 3, 5, 24, 25, 26, 777, 16960, 16963):
        x = (rng.standard_normal(n) + 1j * rng.standard_normal(n)).astype(np.complex64)
        assert oracle.mf(x, 0).tobytes() == oracle.mf(x, 3).tobytes(), n
    from oracle.pyoracle import Oracle
    for adc, ntaps in ((1000000, 12), (1000000, 13), (4000000, 50)):
        o = Oracle(adc_rate=adc, ntaps=ntaps)
        x = (rng.standard_normal(5000) + 1j * rng.standard_normal(5000)).astype(np.complex64)
        assert o.mf(x, 0).tobytes() == o.mf(x, 3).tobytes(), (adc, ntaps)


def test_independent_segments_have_their_own_stop_rule():
    """continuous=0: a segment is a reference run with fresh blocks and reader_state, so the unique-tag stop rule
    (gate_impl.cc:101-104) sees only the segment's own tags; the global tag map is for reporting only"""
    from gen2_uhf_rfid_reader_b200 import abi
    from oracle.pyoracle import Oracle
    o = Oracle(max_tags=1)
    recs = np.zeros((3, 4), dtype=abi.RESULT_DTYPE)
    for s in range(3):
        for k in range(4):
            recs[s, k]["kind"] = k & 1
            recs[s, k]["crc_ok"] = 1 if k & 1 else -1
            recs[s, k]["tag_id"] = 10 * s + k      # every EPC a different tag: 2 per segment, 6 globally
    counts = np.full(3, 4, dtype=np.int32)
    st = o.reduce_stats(recs, counts, False)
    # per segment: 2 EPC windows, the second one makes 2 unique tags > max_tags = 1 -> stop AFTER it; all 12 windows count
    assert st.n_windows == 12 and st.n_epc_correct == 6 and st.n_unique_tags == 6
    st_c = o.reduce_stats(recs, counts, True)
    # one continuous run: stops after the second unique tag, i.e. after 4 windows
    assert st_c.n_windows == 4 and st_c.n_epc_correct == 2


def test_crc_known_answers(oracle):
    assert oracle.query_bits(0) == "1000000000000000010000"   # file_sink content / SURVEY Appendix B
    assert oracle.query_bits(4) == "1000000000000010011101"
    assert "".join(map(str, synth.query_bits(0))) == oracle.query_bits(0)
    assert "".join(map(str, synth.query_bits(4))) == oracle.query_bits(4)
    frame = bytes.fromhex("3000300833b2ddd90140000000276d3e")  # the recorded tag's PC+EPC+CRC
    assert oracle.crc16(frame[:14]) == 0x6D3E and oracle.crc16_ok(frame) == 1
    assert synth.crc16_gen2(frame[:14]) == 0x6D3E
    bad = bytearray(frame)
    bad[5] ^= 1
    assert oracle.crc16_ok(bytes(bad)) == 0


def test_cabsf_is_double_sqrt(oracle):
    rng = np.random.default_rng(0)
    x = (rng.standard_normal(20000) * 10 ** rng.uniform(-3, 2, 20000)).astype(np.float32)
    y = (rng.standard_normal(20000) * 10 ** rng.uniform(-3, 2, 20000)).astype(np.float32)
    want = np.sqrt(x.astype(np.float64) ** 2 + y.astype(np.float64) ** 2).astype(np.float32)
    got = np.array([oracle.cabsf(float(a), float(b)) for a, b in zip(x, y)], dtype=np.float32)
    assert got.tobytes() == want.tobytes()


@pytest.mark.parametrize("adc,exp", [(1000000, (5, 5.0, 48, 2, 50, 24, 125, 685)), (2000000, (10, 10.0, 96, 4, 100, 48, 250, 1370)),
                                     (4000000, (20, 20.0, 192, 9, 200, 96, 500, 2740)), (6000000, (30, 30.0, 288, 14, 300, 144, 750, 4110)),
                                     (8000000, (40, 40.0, 384, 19, 400, 192, 1000, 5480))])
def test_rate_sweep_derived_counts(adc, exp):
    """SURVEY.md Appendix A.6 (evaluated there with the reference's own expressions)"""
    from oracle.pyoracle import Oracle
    c = Oracle(adc_rate=adc).cfg
    assert (c.n_tag_bit_i, c.n_tag_bit_f, c.n_T1, c.n_PW, c.win_length, c.dc_length, c.len_rn16, c.len_epc) == exp


def test_empty_and_short_segments(oracle):
    cap = synth.make_capture(2, seed=1)
    iq = cap["iq"].numpy()
    segs = abi.make_segments([0, 5, 100, 0], [0, 3, 4, 700])
    recs, counts, _ = oracle.decode_segments(iq, segs, max_per_seg=2)
    assert counts.tolist() == [0, 0, 0, 0]
