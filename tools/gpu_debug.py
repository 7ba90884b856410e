#!/usr/bin/env python
"""Developer aid: quick parity probe of the CUDA path against the oracle on a GPU box (verbose diffs)."""
import json
import lzma
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from gen2_uhf_rfid_reader_b200 import abi, capi, synth  # noqa: E402
from oracle.pyoracle import Oracle  # noqa: E402


def diff(name, got, ref, n_got, n_ref):
    ok = True
    if n_got != n_ref:
        print("  %s: window count %s vs ref %s" % (name, n_got, n_ref))
        ok = False
    m = min(len(got), len(ref))
    for f in ref.dtype.names:
        a, b = got[f][:m], ref[f][:m]
        bad = np.nonzero((a != b).reshape(m, -1).any(axis=1))[0]
        if bad.size:
            ok = False
            print("  %s: field %-10s differs in %d/%d records, first %d: got %s ref %s" %
                  (name, f, bad.size, m, bad[0], a[bad[0]], b[bad[0]]))
    print("  %s: %s" % (name, "BIT-EXACT" if ok else "MISMATCH"))
    return ok


def main():
    import torch
    print(torch.cuda.get_device_name(0))
    rx = capi.Gen2Rx()
    O = Oracle()
    iq = np.frombuffer(lzma.decompress(open(os.path.join(ROOT, "tests/golden/file_source_test_head.c64.xz"), "rb").read()),
                       dtype=np.complex64)
    # the reference's records on this head of the recording: the first windows of its run on the whole file
    n_head = json.load(open(os.path.join(ROOT, "tests/golden/cfg1_head_ref_stats.json")))["n_windows"]
    golden = np.load(os.path.join(ROOT, "tests/golden/cfg1_ref_records.npy"))[:n_head]
    allok = True

    print("[1] synthetic 64 segments, capture mode")
    cap = synth.make_capture(64, seed=11)
    siq = cap["iq"].numpy()
    t = time.time()
    recs, counts = rx.decode_capture_host(siq, cap["segments"], max_windows=4)
    print("  gpu call %.3f s" % (time.time() - t))
    orec, ocnt, _ = O.decode_segments(siq, cap["segments"], max_per_seg=4)
    print("  counts gpu", counts[:8], "ref", ocnt[:8])
    allok &= diff("synthetic", recs.reshape(-1), orec.reshape(-1), counts.sum(), ocnt.sum())

    print("[2] cfg1 file_source_test as one continuous segment, capture mode")
    segs = abi.make_segments([0], [iq.size])
    t = time.time()
    recs, counts = rx.decode_capture_host(iq, segs, max_windows=256)
    print("  gpu call %.3f s, windows %d" % (time.time() - t, counts[0]))
    allok &= diff("cfg1", recs[0, :counts[0]], golden, counts[0], len(golden))
    st = rx.reduce_stats(recs, counts, True)
    print("  stats: queries %d round %d epc_ok %d tags %s" % (st.n_queries_sent - 1, st.cur_inventory_round,
                                                             st.n_epc_correct, st.tag_map()))

    print("[3] block mode: mf_work / gate_work / decoder_work")
    y_ref = O.mf(iq)
    rx2 = capi.Gen2Rx()
    ys = []
    for c0 in range(0, 200000, 33333):
        ys.append(rx2.mf_work(iq[c0:min(200000, c0 + 33333)]))
    y = np.concatenate(ys)
    print("  mf_work bit-exact:", y.tobytes() == y_ref[:y.size].tobytes(), y.size)
    g = O.gate(y_ref, want_windows=True)
    rx3 = capi.Gen2Rx()
    pos, wins, cur, seek, nwin = 0, [], [], 1, 0
    while pos < y_ref.size and nwin < 6:
        r = rx3.gate_work(y_ref[pos:pos + 4096], seek=seek)
        seek = 0
        pos += r["consumed"]
        cur.append(r["out"])
        if r["closed"]:
            w = np.concatenate(cur)
            cur = []
            wins.append(w)
            nwin += 1
            seek = 2 if (nwin & 1) else 1
    for k, w in enumerate(wins):
        L = rx.len_epc if (k & 1) else rx.len_rn16
        same = w.tobytes() == g["windows"][k][:L].tobytes()
        rec, bits = rx3.decoder_work(k & 1, w)
        ref = O.decode_window(k & 1, w)
        f_ok = all(rec[f].tobytes() == ref[f].tobytes() for f in ("sync_index", "score", "h_re", "h_im", "T", "crc_ok", "tag_id", "bits"))
        print("  window %d: gate %s decoder %s" % (k, "ok" if same else "DIFF", "ok" if f_ok else "DIFF"))
        allok &= same and f_ok
    print("ALL OK" if allok else "FAILURES")


if __name__ == "__main__":
    main()
