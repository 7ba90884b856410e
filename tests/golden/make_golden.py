#!/usr/bin/env python
"""Regenerates tests/golden/* from a checkout of the reference (nkargas/Gen2-UHF-RFID-Reader).

  python tests/golden/make_golden.py REFERENCE_ROOT     (oracle/_ref must have been built from the same checkout:
                                                         GEN2_REFERENCE_ROOT=REFERENCE_ROOT oracle/build_ref.sh)

  file_source_test_head.c64.xz  the first HEAD_SAMPLES samples of the reference's recorded RX capture
                            (gr-rfid/misc/data/file_source_test, 1,247,958 complex64 @ 2 MS/s), xz-compressed: the cfg1
                            parity input.  The whole recording does not compress below 3 MB (sc16 noise); the head
                            holds 15 complete inventory rounds, the one failed round and the stray burst at its start.
  file_sink_commands.json   Query / ACK bit strings decoded from the reference author's committed TX output
                            gr-rfid/misc/data/file_sink (PIE: data0 = 24 samples fall-to-fall, data1 = 48;
                            reader_impl.cc:51-71,84-125) -- 72 Queries and 71 ACKs whose payloads are the
                            RN16s the reference decoded on that run (SURVEY.md Appendix B)
  readme_expected.txt       the known-answer block of README.md:46-53
  cfg1_ref_records.npy      rfid_b200_window_result records produced by oracle/_ref (the reference's own
                            blocks) on the whole recording; cfg1_ref_stats.json the READER_STATS + print_results text
  cfg1_q4_*.                the same with FIXED_Q = 4
  cfg1_head_ref_stats.json  the reference run on the head: its records are the first n_windows of cfg1_ref_records.npy
                            (checked here), plus READER_STATS, print_results text and the TX commands it sent;
                            cfg1_q4_head_ref_stats.json the same with FIXED_Q = 4
  reference_outputs.npz     what oracle/_ref computes in the remaining comparisons of the test suite: records of the
                            synthetic captures in SYNTH_CASES and the reader block's TX envelope for READER_SCRIPTS
"""
import hashlib
import json
import lzma
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

HEAD_SAMPLES = 300000

# synthetic captures decoded by the reference (FIXED_Q = 0 build) as independent segments (max 4 windows each):
# (n_segments, seed, make_capture keywords)
SYNTH_CASES = [(48, 21, dict(n_tags=1)), (48, 21, dict(n_tags=0)), (48, 21, dict(n_tags=6, fixed_q=2)),
               (48, 21, dict(n_tags=1, noise_sigma=0.02)), (40, 5, dict())]


def synth_key(n, seed, kw):
    return "synth_%d_seed%d" % (n, seed) + "".join("_%s%s" % (k, v) for k, v in sorted(kw.items()))


def rn16_bits(rn16s):
    rn16s = np.asarray(rn16s, dtype=np.int64)
    return ((rn16s[:, None] >> np.arange(15, -1, -1)[None, :]) & 1).astype(np.float32)


def tx_script_rn16s():
    """RN16s of the TX synthesiser comparison: random, with the first RN16 of the author's TX capture and all data-1"""
    rn16s = np.random.default_rng(11).integers(0, 65536, size=12)
    rn16s[0], rn16s[1] = 0x0579, 0xFFFF
    return rn16s


# scripted runs of the reader block (gen2flow_reader_script): name -> (fixed_q, RN16 bits [n, 16], dac_rate)
READER_SCRIPTS = {
    "reader_tx_dac1000000": (0, rn16_bits(tx_script_rn16s()), 1000000),
    "reader_tx_dac2000000": (0, rn16_bits(tx_script_rn16s()), 2000000),
    "reader_tx_q4": (4, np.zeros((2, 16), dtype=np.float32), 1000000),
    "reader_tx_random9": (0, np.random.default_rng(3).integers(0, 2, size=(9, 16)).astype(np.float32), 1000000),
}


def iq_digest(iq):
    return hashlib.sha256(np.ascontiguousarray(iq).tobytes()).hexdigest()


def decode_pie(tx):
    """TX envelope (0/1 floats @1 MS/s) -> list of (kind, bitstring)."""
    lvl = tx > 0.5
    fall = np.nonzero(lvl[:-1] & ~lvl[1:])[0] + 1   # first low sample of each pulse
    # group falls into commands: gaps > 400 samples separate commands
    cmds, cur = [], [fall[0]]
    for a, b in zip(fall[:-1], fall[1:]):
        if b - a > 400:
            cmds.append(cur)
            cur = []
        cur.append(b)
    cmds.append(cur)
    out = []
    for c in cmds:
        d = np.diff(c)
        iv = list(d)
        # fall-to-fall intervals: delimiter->data0 low = 24, RTcal = 72, TRcal = 200 (Query only),
        # then one interval per bit (every PIE symbol ends with its low pulse): 24 = '0', 48 = '1'
        assert iv[0] == 24 and iv[1] == 72, iv[:4]
        k = 2
        kind = "framesync"
        if iv[k] == 200:
            kind = "preamble"
            k += 1
        assert all(x in (24, 48) for x in iv[k:]), iv
        bits = "".join("1" if x == 48 else "0" for x in iv[k:])
        out.append((kind, bits))
    return out


def _stats_json(r):
    s = r["stats"]
    return {"text": r["text"], "n_queries_sent": s.n_queries_sent,
            "cur_inventory_round": s.cur_inventory_round, "cur_slot_number": s.cur_slot_number,
            "n_epc_correct": s.n_epc_correct, "tag_reads": {str(k): v for k, v in s.tag_map().items()},
            "n_windows": r["n_windows"]}


def main(ref_root):
    from gen2_uhf_rfid_reader_b200 import synth
    from oracle.refflow import RefFlow
    src = os.path.join(ref_root, "gr-rfid/misc/data/file_source_test")
    raw = open(src, "rb").read()
    iq = np.frombuffer(raw, dtype=np.complex64)
    head = iq[:HEAD_SAMPLES]
    with open(os.path.join(HERE, "file_source_test_head.c64.xz"), "wb") as f:
        f.write(lzma.compress(head.tobytes(), preset=9 | lzma.PRESET_EXTREME))

    sink = np.fromfile(os.path.join(ref_root, "gr-rfid/misc/data/file_sink"), dtype=np.complex64).real
    amp = sink.max()
    cmds = decode_pie(sink / amp)
    queries = [b for k, b in cmds if k == "preamble"]
    acks = [b for k, b in cmds if k == "framesync"]
    rn16 = ["%04x" % int(b[2:], 2) for b in acks]
    json.dump({"amplitude": float(amp), "n_lead_cw": int(np.argmax(sink / amp < 0.5)),
               "queries": queries, "acks": acks, "rn16": rn16},
              open(os.path.join(HERE, "file_sink_commands.json"), "w"), indent=1)

    readme = open(os.path.join(ref_root, "README.md")).read().splitlines()
    open(os.path.join(HERE, "readme_expected.txt"), "w").write("\n".join(readme[45:53]) + "\n")

    for q, tag in ((0, "cfg1"), (4, "cfg1_q4")):
        r = RefFlow(q).run_stream(iq)
        np.save(os.path.join(HERE, tag + "_ref_records.npy"), r["records"])
        json.dump(_stats_json(r), open(os.path.join(HERE, tag + "_ref_stats.json"), "w"), indent=1)
        h = RefFlow(q).run_stream(head, want_tx=True)
        n = h["n_windows"]
        assert h["records"].tobytes() == r["records"][:n].tobytes(), "head records are not a prefix of the full run"
        for chunk in (257, 100000):
            assert RefFlow(q).run_stream(head, chunk=chunk)["records"].tobytes() == h["records"].tobytes(), chunk
        tx = decode_pie(h["tx"])
        hs = _stats_json(h)
        hs.update(samples=HEAD_SAMPLES, sha256=iq_digest(head), tx_samples=int(h["tx"].size),
                  tx_queries=[b for k, b in tx if k == "preamble"], tx_acks=[b for k, b in tx if k == "framesync"])
        json.dump(hs, open(os.path.join(HERE, tag + "_head_ref_stats.json"), "w"), indent=1)

    out = {}
    for n, seed, kw in SYNTH_CASES:
        cap = synth.make_capture(n, seed=seed, **kw)
        cap_iq = cap["iq"].numpy()
        recs, counts, _ = RefFlow(0).run_segments(cap_iq, cap["segments"], max_per_seg=4)
        key = synth_key(n, seed, kw)
        out[key + "_records"] = recs
        out[key + "_counts"] = counts
        out[key + "_sha256"] = np.array(iq_digest(cap_iq))
    for name, (q, bits, dac) in READER_SCRIPTS.items():
        tx, nq = RefFlow(q).reader_script(bits, dac_rate=dac)
        out[name] = tx
        out[name + "_queries"] = np.array(nq)
    np.savez_compressed(os.path.join(HERE, "reference_outputs.npz"), **out)
    print("golden regenerated:", sorted(os.listdir(HERE)))


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    main(sys.argv[1])
