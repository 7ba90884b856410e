#!/usr/bin/env python
"""Developer aid (GPU box): where the time of bench.py cfg2's step goes.

Same inputs as bench.py cfg2 (4 captures of 1000 segments, seeds 1234 + 17 b, records into 8 slots, one decode_capture
per step on the current stream).  Prints, from one process:
  * the card, its SM clock and power limit;
  * ms_per_step from CUDA events around the timed loop, with kernel timing on and off, and kernel_time per launch;
  * a per-launch timeline from a build with RFID_B200_PHASE_PROFILE (per-CTA %globaltimer stamps, one window tap per
    launch): each launch's first CTA start against the previous launch's last CTA end (negative = the launches overlap),
    and the spread of the CTAs' last-decode times; and the smallest non-zero difference between two stamps (the
    resolution of %globaltimer).
usage: python tools/step_timeline.py [--steps 20] [--warmup 3] [--nseg 1000]"""
import argparse
import os
import subprocess
import sys
import tempfile

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from gen2_uhf_rfid_reader_b200 import build, capi, synth  # noqa: E402

MAX_WINDOWS = 4


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,clocks.sm,clocks.max.sm,power.limit", "--format=csv,noheader",
                        "-i", "0"], capture_output=True, text=True)
    return q.stdout.strip() or "nvidia-smi: %s" % q.stderr.strip()


def profile_context(tmp):
    """a second context on a library built with RFID_B200_PHASE_PROFILE (in a temporary directory)"""
    lib = os.path.join(tmp, "librfid_b200_prof.so")
    subprocess.check_call(["nvcc"] + build.NVCC_FLAGS + ["-DRFID_B200_PHASE_PROFILE", "-o", lib,
                                                         os.path.join(build.CSRC, "rfid_b200.cu")])
    saved, env = capi._lib, os.environ.get("RFID_B200_LIB")
    capi._lib, os.environ["RFID_B200_LIB"] = None, lib
    try:
        return capi.Gen2Rx()
    finally:
        capi._lib = saved
        if env is None:
            del os.environ["RFID_B200_LIB"]
        else:
            os.environ["RFID_B200_LIB"] = env


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--nseg", type=int, default=1000)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    print("card (name, SM clock, max SM clock, power limit):", card())
    nseg = args.nseg
    caps, seg_dev = [], None
    for b in range(4):
        cap = synth.make_capture(nseg, seed=1234 + 17 * b, device=dev)
        caps.append(cap["iq"])
        if seg_dev is None:
            seg_dev = capi.segments_to_device(cap["segments"], dev)
    nslots = 8
    res = torch.zeros((nslots, nseg * MAX_WINDOWS, 64), dtype=torch.uint8, device=dev)
    cnt = torch.zeros((nslots, nseg), dtype=torch.int32, device=dev)
    stream = torch.cuda.current_stream(dev)

    def loop(rx, timing, taps=None):
        for i in range(args.warmup):
            rx.decode_capture(caps[i % 4], seg_dev, MAX_WINDOWS, res[i % nslots], cnt[i % nslots], stream)
        torch.cuda.synchronize()
        if timing:
            rx.enable_kernel_timing(True)
            rx.kernel_time(reset=True)
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record(stream)
        for i in range(args.steps):
            if taps is not None:
                rx.set_window_tap(taps[i])
            rx.decode_capture(caps[(args.warmup + i) % 4], seg_dev, MAX_WINDOWS, res[i % nslots], cnt[i % nslots], stream)
        ev1.record(stream)
        torch.cuda.synchronize()
        k_ms, k_n = rx.kernel_time(reset=True)
        rx.enable_kernel_timing(False)
        if taps is not None:
            rx.set_window_tap(None)
        return ev0.elapsed_time(ev1) / args.steps, (k_ms / k_n if k_n else float("nan")), k_n

    rx = capi.Gen2Rx()
    print("\nms_per_step (CUDA events around %d steps after %d warm-up steps)" % (args.steps, args.warmup))
    for rep in range(2):
        for timing in (True, False):
            ms, k_ms, k_n = loop(rx, timing)
            print("  kernel timing %-3s  ms_per_step %.4f" % ("on" if timing else "off", ms) +
                  ("   kernel_time %.4f ms per launch over %d launches" % (k_ms, k_n) if timing else ""))

    with tempfile.TemporaryDirectory() as tmp:
        prx = profile_context(tmp)
        ncta = (nseg + 6) // 7
        taps = [torch.zeros(512 * 8 + 2 * ncta + 64, dtype=torch.int64, device=dev) for _ in range(args.steps)]
        ms, _, _ = loop(prx, False, taps)
        prx.close()
    ct = np.stack([t[512 * 8: 512 * 8 + 2 * ncta].cpu().numpy().reshape(ncta, 2) for t in taps]).astype(np.int64)
    starts, ends = ct[:, :, 0], ct[:, :, 1]
    t0 = starts[0].min()
    print("\nper-launch timeline (profile build, ms_per_step %.4f; us from the first CTA start of the first timed launch)" % ms)
    print("launch | first CTA start  last CTA start | last decode: first  median  last | start - previous last decode")
    prev_end = None
    gaps = []
    for i in range(args.steps):
        s, e = (starts[i] - t0) / 1e3, (ends[i] - t0) / 1e3
        gap = s.min() - prev_end if prev_end is not None else float("nan")
        if prev_end is not None:
            gaps.append(gap)
        print("%6d | %15.2f %15.2f | %18.2f %7.2f %6.2f | %+8.2f" % (i, s.min(), s.max(), e.min(), np.median(e), e.max(), gap))
        prev_end = e.max()
    spread = [(ends[i].max() - np.median(ends[i])) / 1e3 for i in range(args.steps)]
    dur = [(ends[i].max() - starts[i].min()) / 1e3 for i in range(args.steps)]
    print("median: start - previous last decode %+.2f us, launch span %.2f us, last decode - median decode %.2f us"
          % (np.median(gaps), np.median(dur), np.median(spread)))
    stamps = np.unique(np.concatenate([starts.ravel(), ends.ravel()]))
    print("%%globaltimer: smallest non-zero difference between two of %d stamps: %d ns" % (stamps.size, int(np.diff(stamps).min())))


if __name__ == "__main__":
    main()
