"""CPU tests of host-side logic: synthetic generator, segment sharding, the world-size-2 gather (gloo)."""
import os
import socket
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT
from gen2_uhf_rfid_reader_b200 import abi, shard, synth


def test_synth_is_deterministic_and_shard_invariant():
    a = synth.make_capture(12, seed=9)
    b = synth.make_capture(12, seed=9)
    assert torch.equal(a["iq"], b["iq"])
    part = synth.make_capture(4, seed=9, first_segment=8)
    L = a["truth"]["segment_len"]
    # per-segment protocol content (RN16, EPC, timing) depends only on (seed, segment id)
    assert (part["truth"]["rn16"] == a["truth"]["rn16"][8:]).all()
    assert (part["truth"]["epc"] == a["truth"]["epc"][8:]).all()
    assert L == 16960 and a["iq"].numel() == 12 * L
    assert (a["segments"]["offset"] == np.arange(12) * L).all()


def test_synth_collisions_q4():
    cap = synth.make_capture(64, seed=2, fixed_q=4, n_tags=8)
    t = cap["truth"]
    assert t["is_query"].sum() == 4 and t["is_query"][::16].all()
    per_round = t["n_replies"].reshape(4, 16).sum(axis=1)
    assert (per_round == 8).all()          # every tag answers in exactly one slot of its round
    assert (t["n_replies"] >= 2).any()     # with 8 tags in 16 slots some slot collides


def test_epc_frames_have_valid_crc():
    fr = synth.make_epc_frames(np.arange(24, dtype=np.uint8).reshape(2, 12))
    for f in fr:
        assert synth.crc16_gen2(bytes(f[:14])) == (int(f[14]) << 8 | int(f[15]))


@pytest.mark.parametrize("n,w", [(1000, 1), (1000, 8), (7, 4), (3, 8), (0, 2)])
def test_shard_ranges_partition(n, w):
    r = [shard.shard_range(n, k, w) for k in range(w)]
    assert r[0][0] == 0 and r[-1][1] == n
    assert all(a[1] == b[0] for a, b in zip(r, r[1:]))
    assert max(e - b for b, e in r) <= shard.max_shard(n, w)


def _gloo_worker(rank, world, port, n_seg, out_q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    import torch.distributed as dist
    sys.path.insert(0, ROOT)
    from oracle.pyoracle import Oracle  # the checker stands in for the GPU decode in this CPU test
    dist.init_process_group("gloo", rank=rank, world_size=world)
    cap_all = synth.make_capture(n_seg, seed=31)
    b, e = shard.shard_range(n_seg, rank, world)
    L = cap_all["truth"]["segment_len"]
    iq = cap_all["iq"].numpy()[b * L:e * L]
    segs = abi.make_segments(np.arange(e - b) * L, [L] * (e - b))
    recs, counts, _ = Oracle().decode_segments(iq, segs, max_per_seg=2)
    shard.renumber_segments(recs, b)
    res_t = torch.from_numpy(recs.reshape(-1).view(np.uint8).reshape(-1, 64).copy())
    cnt_t = torch.from_numpy(counts.copy())
    g_res, g_cnt = shard.gather_records(res_t, cnt_t, n_seg, 2)
    if rank == 0:
        out_q.put((g_res.numpy().tobytes(), g_cnt.numpy().tobytes()))
    dist.barrier()
    dist.destroy_process_group()


def test_gather_records_world2_gloo():
    """N>1 path on CPU: two ranks decode disjoint shards, one all-gather, rank 0 sees the single-process result"""
    import torch.multiprocessing as mp
    n_seg = 5   # odd => unequal shards exercise the padding
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, n_seg, q)) for r in range(2)]
    for p in procs:
        p.start()
    res_b, cnt_b = q.get(timeout=120)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    from oracle.pyoracle import Oracle
    cap = synth.make_capture(n_seg, seed=31)
    recs, counts, _ = Oracle().decode_segments(cap["iq"].numpy(), cap["segments"], max_per_seg=2)
    got = np.frombuffer(res_b, dtype=abi.RESULT_DTYPE).reshape(n_seg, 2)
    assert np.frombuffer(cnt_b, dtype=np.int32).tolist() == counts.tolist()
    for f in recs.dtype.names:
        assert got[f].tobytes() == recs[f].tobytes(), f


def test_reader_block_matches_reference_sample_for_sample(ref_outputs):
    """this repo's reader block (Gen2 logic + PIE generator, host C++) vs the reference's, scripted on CPU:
    START, Query/QueryRep alternating, ACK(RN16), CW -- identical TX envelope and query count"""
    from make_golden import READER_SCRIPTS
    from oracle import refflow
    mine = refflow.B200Flow()
    _, bits, _ = READER_SCRIPTS["reader_tx_random9"]
    assert np.array_equal(bits, np.random.default_rng(3).integers(0, 2, size=(9, 16)).astype(np.float32))
    a, na = ref_outputs["reader_tx_random9"], int(ref_outputs["reader_tx_random9_queries"])
    b, nb = mine.reader_script(bits)
    assert na == nb == 9
    assert a.size == b.size and np.array_equal(a, b)
    # and the Query it sends is the one in the reference author's TX capture
    import json
    from conftest import GOLDEN
    from make_golden import decode_pie
    cmds = decode_pie(b)
    gold = json.load(open(os.path.join(GOLDEN, "file_sink_commands.json")))
    assert [c for k, c in cmds if k == "preamble"][0] == gold["queries"][0]
    acks = [c for k, c in cmds if k == "framesync" and len(c) == 18]
    assert acks[0] == "01" + "".join(str(int(x)) for x in bits[0])


def test_constant_division_sequence_is_exact_for_every_float():
    """the 3-instruction multiply-correct division used by the kernels equals IEEE x/d for EVERY binary32
    mantissa, for every divisor the host marks as 'fast' (csrc/rfid_b200.cu kVerifiedDivisors + 6, 19)"""
    import re
    import subprocess
    src = open(os.path.join(ROOT, "gen2_uhf_rfid_reader_b200", "csrc", "rfid_b200.cu")).read()
    m = re.search(r"kVerifiedDivisors\[\] = \{([^}]*)\}", src)
    divs = sorted(set(int(x) for x in m.group(1).split(",")) | {6, 19})
    exe = "/tmp/verify_constdiv_%d" % os.getpid()
    subprocess.check_call(["gcc", "-O2", "-ffp-contract=off", "-o", exe,
                           os.path.join(ROOT, "tools", "micro", "verify_constdiv.c"), "-lm"])
    out = subprocess.run([exe] + [str(d) for d in divs], capture_output=True, text=True)
    os.unlink(exe)
    assert out.returncode == 0, out.stdout
    assert out.stdout.count(": 0 mismatches") == len(divs)


# ------------------------------------------------------------------ capture ingest: segmentation rule (CPU model)
def test_segmenter_rule_on_golden_recording(cfg1_iq, cfg1_golden):
    """the CW-gap rule on the reference's recording: 16 Queries + 16 ACKs found, one stray burst rejected,
    every golden window lies inside exactly the segment that holds its command"""
    import segmenter_model as sm
    pos, pulses = sm.bursts(cfg1_iq)
    assert sorted(set(pulses.tolist())) == [3, 21, 26]          # stray pulses, ACK (21), Query (26)
    segs, cmd = sm.segment_table(cfg1_iq)
    assert len(cmd) == 32 and len(segs) == 16
    assert all(off % 5 == 0 for off, _ in segs) and segs[0][0] == 0
    assert segs[-1][0] + segs[-1][1] == cfg1_iq.size
    opens = cfg1_golden["open_index"].astype(np.int64) * 5      # raw index of every golden window
    ends = opens + cfg1_golden["length"].astype(np.int64) * 5
    assert len(cfg1_golden) == 31
    for k in range(31):
        off, ln = segs[k // 2]
        assert off < opens[k] and ends[k] <= off + ln, k
        # the window belongs to command k: it opens after that command and before the next one
        assert cmd[k] < opens[k] and (k + 1 >= len(cmd) or ends[k] < cmd[k + 1])


def test_segmenter_rule_on_synthetic_capture():
    import segmenter_model as sm
    cap = synth.make_capture(24, seed=3)
    iq = cap["iq"].numpy()
    segs, cmd = sm.segment_table(iq)
    assert len(segs) == 24 and len(cmd) == 48
    gen = cap["segments"]
    for (off, ln), g in zip(segs, gen):
        # segmenter's cut lies in the generator's lead-in CW of the same round
        assert int(g["offset"]) <= off + 1200 and off < int(g["offset"]) + int(g["length"])
