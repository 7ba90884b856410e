#!/usr/bin/env python
"""bench.py -- MSamples/s of raw I/Q through matched filter -> gate -> tag_decoder.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config cfg2|cfg3|cfg4|cfg5]
                  [--dump-outputs DIR]

Default workload = BASELINE.json configs[1] ("cfg2"): synthetic 40 kHz-BLF FM0 I/Q @ 2 MS/s, 1000 queries
(= 1000 inventory-round segments of 16,960 raw samples), 1 tag, per GPU.  One *step* = one pass of the hot path
over one such capture.  `value` is timed with the captures already resident in HBM; `e2e` goes through the
host-pointer C-ABI call with pinned host buffers (H2D of the capture and D2H of the records inside the timed
region).  Weak scaling: every rank decodes its own shard of the global segment table; the one collective is a
single all-gather of the decoded records (window counts travel in the same block) of all K steps at the end
of the timed region.

Other BASELINE.json configurations (measurement runs; the driver's line stays cfg2):
  cfg3  100,000 inventory rounds in total (1.696e9 raw samples), FIXED_Q=0, sharded over the GPUs ("strong")
  cfg4  FIXED_Q=4: 10,000 rounds x 16 slots = 160,000 slot segments with 8 tags (empty, single and collided slots)
  cfg5  raw-rate sweep 1 / 2 / 4 / 6 / 8 MS/s (decimation 5, ntaps = rate / (2 BLF)): kernel GB/s vs the HBM roofline

--dump-outputs DIR writes what the last timed step computed (window records and counts, see dump_outputs) as
DIR/<name>.npy; the workload is generated from fixed seeds, so two builds run with the same arguments can be
compared output for output.

--impl reference times the reference's own CPU implementation (oracle/_ref: its blocks compiled unchanged, behind
the canonical matched filter -- GNU Radio's own FIR is not in the reference tree) on all usable host cores over
the same workload (a bounded sample of it for cfg3 / cfg4).
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SEG_US = 8480.0
NBUF = 4          # cfg2: distinct captures cycled through so every step reads data that is not in L2
MAX_WINDOWS = 2
METRIC = "MSamples/s I/Q through gate->tag_decoder"
BLF = 40000

CONFIGS = {
    "cfg2": dict(rounds=1000, fixed_q=0, n_tags=1, adc_rate=2_000_000, ntaps=25, scaling="weak", nbuf=NBUF,
                 text="cfg2: synthetic 40kHz-BLF FM0 I/Q @2Msps, %(rounds)d queries (inventory rounds) x %(seg_len)d raw samples, 1 tag, per GPU"),
    "cfg3": dict(rounds=100000, fixed_q=0, n_tags=1, adc_rate=2_000_000, ntaps=25, scaling="strong", nbuf=1,
                 text="cfg3: synthetic %(total)d inventory rounds in total (%(total_samples).4g raw samples: 100k rounds fixed, "
                      "BASELINE's '1e9 samples' does not fit 100k physically valid rounds), FIXED_Q=0, rounds sharded over the GPUs"),
    "cfg4": dict(rounds=10000, fixed_q=4, n_tags=8, adc_rate=2_000_000, ntaps=25, scaling="weak", nbuf=1,
                 text="cfg4: FIXED_Q=4, %(rounds)d rounds x 16 slots = %(nseg)d slot segments x %(seg_len)d raw samples, 8 tags "
                      "(empty, singly occupied and collided slots), per GPU"),
}
SWEEP_RATES = [1_000_000, 2_000_000, 4_000_000, 6_000_000, 8_000_000]
DUMP_BYTES = 60_000_000     # --dump-outputs payload: with the .npy headers below 64 MB however counted


def dump_outputs(out_dir, recs, counts, prefix="", extra=None, limit=DUMP_BYTES):
    """Writes decoded window records (RESULT_DTYPE[nseg, max_windows]) and window counts (int32[nseg]) as
    out_dir/<prefix><name>.npy: counts.npy and one records_<field>.npy per record field, integer fields as float64,
    float fields and the bit bytes as float32 (all exact).  `extra` maps names to further per-segment arrays.
    Above `limit` bytes in all, a fixed seeded sample of the segments is written, their indices in segment_index.npy."""
    def arrays(sel):
        out = {"counts": counts[sel].astype(np.float64)}
        for name in recs.dtype.names:
            a = recs[name][sel]
            out["records_" + name] = a.astype(np.float64 if a.dtype.kind == "i" else np.float32)
        for name, a in (extra or {}).items():
            out[name] = np.asarray(a)[sel].astype(np.float64)
        return out

    nseg = counts.size
    per_seg = sum(a.nbytes for a in arrays(slice(0, 1)).values())
    if nseg * per_seg <= limit:
        out = arrays(slice(None))
    else:
        idx = np.sort(np.random.default_rng(0).choice(nseg, limit // (per_seg + 8), replace=False))
        out = arrays(idx)
        out["segment_index"] = idx.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, prefix + name + ".npy"), a)


def hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured"
        except Exception:
            pass
    return 6650.0, "fallback"


class ClockSampler:
    """SM clock / throttle reasons sampled through NVML from a background thread (every ~0.5 ms) so that even a
    millisecond-long timed region gets samples; `window(t0, t1)` summarises the samples taken inside it."""

    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index):
        self.index, self.rows, self.stop_flag, self.th, self.ok = index, [], False, None, False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_sm = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.ok = True
        except Exception:
            self.ok = False

    def start(self):
        if not self.ok:
            return
        self.th = threading.Thread(target=self._run, daemon=True)
        self.th.start()

    def _run(self):
        nv = self.nv
        while not self.stop_flag:
            try:
                mhz = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                try:
                    rs = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    rs = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.rows.append((time.perf_counter(), float(mhz), int(rs)))
            except Exception:
                pass
            time.sleep(0.0004)

    def stop(self):
        self.stop_flag = True
        if self.th:
            self.th.join(timeout=1)

    def window(self, t0, t1):
        if not self.ok:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable"], "samples": 0}
        inside = [r for r in self.rows if t0 <= r[0] <= t1]
        pad = 0.0
        while len(inside) < 3 and pad < 0.2:   # very short region: widen symmetrically, say so
            pad += 0.005
            inside = [r for r in self.rows if t0 - pad <= r[0] <= t1 + pad]
        reasons = set()
        for r in inside:
            for bit, nm in self.REASONS.items():
                if r[2] & bit:
                    reasons.add(nm)
        return {"sm_mhz": float(np.median([r[1] for r in inside])) if inside else None, "sm_max_mhz": self.max_sm,
                "reasons": sorted(reasons), "samples": len(inside), "window_pad_ms": round(pad * 1e3, 1)}


# ----------------------------------------------------------------------------------------- host topology
def host_cores():
    """CPUs this process may actually use: affinity mask, capped by the cgroup CPU quota (a container that sees
    128 logical CPUs but is granted 16 CPUs of time is a 16-core host for this purpose -- more runnable
    processes than that only get throttled)."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    quota = None
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            quota = int(q) / int(p)
    except (OSError, ValueError):
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            p = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / p
        except (OSError, ValueError):
            pass
    if quota:
        n = min(n, max(1, int(quota + 0.5)))
    return max(1, n)


def bind_to_gpu_numa_node(local_rank):
    """Pin this rank (and therefore the pinned host buffers it allocates afterwards, first-touch) to the NUMA node
    its GPU hangs off, so that the end-to-end leg's host<->device copies do not cross the socket interconnect.
    Returns a short description for the bench line; silently does nothing where the topology is not exposed."""
    try:
        import torch
        pr = torch.cuda.get_device_properties(local_rank)
        bus = "%04x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bus).read())
        if node < 0:
            return "numa node not reported"
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        allowed = cpus & set(os.sched_getaffinity(0))
        if not allowed:
            return "numa node %d has no allowed CPUs" % node
        os.sched_setaffinity(0, allowed)
        return "rank bound to NUMA node %d (%d CPUs)" % (node, len(allowed))
    except Exception as e:  # noqa: BLE001 -- topology files are optional
        return "not bound (%s)" % type(e).__name__


# ----------------------------------------------------------------------------------------- reference arm
_G = {}


def _ref_init(kind, fixed_q):
    from oracle import pyoracle, refflow
    _G["flow"] = refflow.RefFlow(fixed_q) if kind == "reference" else pyoracle.Oracle(fixed_q=fixed_q)
    _G["kind"] = kind


def _ref_worker(args):
    seg_bytes, passes, adc_rate, ntaps = args
    from gen2_uhf_rfid_reader_b200 import abi
    segs = np.frombuffer(seg_bytes, dtype=abi.SEGMENT_DTYPE)
    iq = _G["iq"]          # inherited through fork (copy-on-write, never written)
    t, n = 0.0, 0
    for _ in range(passes):
        if _G["kind"] == "reference":
            # timing run: no record buffer, so only the blocks' own work is inside the timer
            _, counts, secs = _G["flow"].run_segments(iq, segs, adc_rate=adc_rate, ntaps=ntaps, max_per_seg=MAX_WINDOWS,
                                                      want_records=False)
        else:
            _, counts, secs = _G["flow"].decode_segments(iq, segs, max_per_seg=MAX_WINDOWS)
        t += secs
        n += int(counts.sum())
    return t, n


def cpu_reference_run(iq_np, segs, steps, warmup, passes_per_step=1, fixed_q=0, adc_rate=2_000_000, ntaps=25, what="cfg2 capture"):
    """Reference CPU implementation on all usable host cores: one process per core over disjoint segment ranges
    (the reference keeps its state in a process global, include/rfid/global_vars.h:146).  Timed by wall
    clock around each step (all processes working), excluding data generation and file I/O."""
    import multiprocessing as mp
    from oracle import refflow
    kind = "reference" if refflow.ref_available(fixed_q) else "port"
    cores = host_cores()
    nseg = segs.size
    _G["iq"] = np.ascontiguousarray(iq_np)
    jobs = []
    for c in range(cores):
        b, e = c * nseg // cores, (c + 1) * nseg // cores
        jobs.append((segs[b:e].copy().tobytes(), passes_per_step, adc_rate, ntaps))
    ctx = mp.get_context("fork")
    times, windows = [], 0
    with ctx.Pool(cores, initializer=_ref_init, initargs=(kind, fixed_q)) as pool:
        for it in range(warmup + steps):
            t0 = time.perf_counter()
            out = pool.map(_ref_worker, jobs, chunksize=1)
            dt = time.perf_counter() - t0
            if it >= warmup:
                times.append(dt)
                windows = sum(o[1] for o in out)
    _G.pop("iq", None)
    n_samples = float(segs["length"].astype(np.float64).sum()) * passes_per_step
    total = sum(times)
    return {"kind": kind, "cores": cores, "ms_per_step": 1e3 * total / max(1, len(times)),
            "value": n_samples * len(times) / total / 1e6, "windows_last_step": windows,
            "sample": "%s: %d segments (%.1f M samples) split over %d processes (= usable CPUs: affinity and cgroup quota; "
                      "os.cpu_count() = %d), %d pass(es) per step, %d steps; the reference's gate / tag_decoder / reader "
                      "blocks compiled unchanged, fresh blocks per segment; matched filter = canonical-order boxcar with every "
                      "block sum formed once, compiler-vectorised (stand-in for GNU Radio's VOLK FIR, which is not in the "
                      "reference tree; about a third of this arm's time)"
                      % (what, nseg, n_samples / passes_per_step / 1e6, cores, os.cpu_count() or 1, passes_per_step, len(times))}


# ----------------------------------------------------------------------------------------- workload
def ntaps_for(adc_rate):
    return max(1, int(round(adc_rate / (2.0 * BLF))))      # half an FM0 symbol (apps/reader.py:65); 12.5 -> 12 at 1 MS/s


def kernel_name(adc_rate, ntaps):
    fs = adc_rate // 5
    if ntaps == 25 and int(250e-6 * fs) <= 128:
        return "rx_pack_kernel<5,5> (matched filter + gate + tag_decoder; segments packed per CTA, shared running-sum warp)"
    if int(250e-6 * fs) <= 128:
        return "rx_fused_split_kernel<5,%d> (one CTA per segment)" % (ntaps // 5 if ntaps % 5 == 0 and ntaps // 5 == 5 else 0)
    return "rx_fused_kernel<5,0> (one CTA per segment, explicit rings)"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="cfg2", choices=["cfg2", "cfg3", "cfg4", "cfg5", "ingest"])
    ap.add_argument("--rounds", type=int, default=None, help="inventory rounds (cfg2/cfg4: per GPU; cfg3: in total)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--generator", default="torch", choices=["torch", "native"],
                    help="workload generator of our arm (cfg2): the torch model (same samples as the CPU reference arm) or the "
                         "library's CUDA closed-loop slot simulator (rfid_b200_sim_capture)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the window records and counts of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps is not None and args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what our timed path computed; the reference arm keeps no records")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.steps is None:
        args.steps = 20 if args.config == "cfg2" else 5

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.config == "cfg5":
        return sweep(args, rank, local_rank, world)
    if args.config == "ingest":
        return ingest(args, rank, local_rank)

    from gen2_uhf_rfid_reader_b200 import abi, synth
    cfg = dict(CONFIGS[args.config])
    if args.rounds is not None:
        cfg["rounds"] = args.rounds
    adc_rate, ntaps, fixed_q, n_tags = cfg["adc_rate"], cfg["ntaps"], cfg["fixed_q"], cfg["n_tags"]
    seg_len = int(round(SEG_US * adc_rate / 1e6))
    slots = 1 << fixed_q
    if cfg["scaling"] == "strong":
        total_seg = cfg["rounds"] * slots
        b = rank * total_seg // world
        e = (rank + 1) * total_seg // world
        nseg, first = e - b, b
        n_global = total_seg
    else:
        nseg = cfg["rounds"] * slots
        first = nseg * rank
        n_global = nseg * world
    fmt = dict(rounds=cfg["rounds"], seg_len=seg_len, nseg=nseg, total=cfg["rounds"], total_samples=float(cfg["rounds"]) * slots * seg_len)
    config = {"workload": cfg["text"] % fmt, "config": args.config, "segments_per_gpu": nseg, "segments_total": n_global,
              "segment_samples": seg_len, "fixed_q": fixed_q, "n_tags": n_tags,
              "l2": "inputs larger than L2: %d distinct capture(s) of %.0f MB per GPU" % (cfg["nbuf"], nseg * seg_len * 8 / 1e6),
              "parallelism": "segments sharded over %d GPU(s), one all-gather of all decoded records (+ window counts, same block) "
                             "at the end of the timed region" % world,
              "generator": args.generator}

    # ------------------------------------------------------------------ reference arm (CPU, rank 0 only)
    if args.impl == "reference":
        if rank != 0:
            return 0
        n_samp = min(nseg, 1000 if fixed_q == 0 else 2048)
        cap = synth.make_capture(n_samp, seed=1234, device="cpu", fixed_q=fixed_q, n_tags=n_tags, adc_rate=adc_rate)
        # each step = 8 passes over the sample (bounded: ~0.05 s per step on a 16-CPU host)
        r = cpu_reference_run(cap["iq"].numpy(), cap["segments"], args.steps, args.warmup, passes_per_step=8, fixed_q=fixed_q,
                              adc_rate=adc_rate, ntaps=ntaps, what="%s sample" % args.config)
        line = {"impl": "reference", "metric": METRIC, "value": r["value"], "unit": "MSamples/s", "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True,
                "scaling": cfg["scaling"], "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
                "cpu_baseline": {"value": r["value"], "unit": "MSamples/s", "cores": r["cores"], "kind": r["kind"],
                                 "sample": r["sample"]},
                "e2e": {"value": r["value"], "unit": "MSamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line))
        return 0

    # ------------------------------------------------------------------ our arm
    import torch
    import torch.distributed as dist
    from gen2_uhf_rfid_reader_b200 import capi
    assert torch.cuda.is_available(), "bench.py --impl ours needs a GPU (there is no CPU fallback)"
    torch.cuda.set_device(local_rank)
    affinity0 = os.sched_getaffinity(0)
    numa = bind_to_gpu_numa_node(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    rx = capi.Gen2Rx(device=local_rank, fixed_q=fixed_q, adc_rate=adc_rate, ntaps=ntaps)
    caps, truths, seg_dev = [], [], None
    for b in range(cfg["nbuf"]):
        if args.generator == "native" and args.config == "cfg2":
            sim = capi.default_sim(seed=1234 + 17 * b, segment_us=SEG_US)
            cap = rx.sim_capture(sim, nseg, first_segment=first, device=dev)
            tr = cap["truth"].cpu().numpy().view(abi.SIM_TRUTH_DTYPE).reshape(-1)
            caps.append(cap["iq"])
            truths.append({"rn16": tr["acked_rn16"].astype(np.int64), "epc": tr["epc"]})
            if seg_dev is None:
                seg_dev = cap["segs"]
                segs_np = cap["segs"].cpu().numpy().view(abi.SEGMENT_DTYPE).reshape(-1)
        else:
            cap = synth.make_capture(nseg, seed=1234 + 17 * b, first_segment=first, device=dev, fixed_q=fixed_q, n_tags=n_tags,
                                     adc_rate=adc_rate)
            caps.append(cap["iq"])
            truths.append(cap["truth"])
            if seg_dev is None:
                segs_np = cap["segments"]
                seg_dev = capi.segments_to_device(segs_np, dev)
    n_raw = caps[0].numel()
    # every step keeps its records on the device; ONE all-gather of all of them closes the timed region (north star: "a
    # single NCCL gather of decoded EPCs at the end").  Records and window counts share one block per step:
    # rows [0, nseg*MAX_WINDOWS) = 64-byte records, the rows after them = the int32 counts.
    nslots = max(min(args.steps, 8), args.warmup)
    cnt_rows = (nseg * 4 + 63) // 64
    block = torch.zeros((nslots, nseg * MAX_WINDOWS + cnt_rows, 64), dtype=torch.uint8, device=dev)
    g_block = torch.empty((world,) + tuple(block.shape), dtype=torch.uint8, device=dev) if world > 1 else None
    stream = torch.cuda.current_stream(dev)
    launches = 0

    def res_of(slot):
        return block[slot, : nseg * MAX_WINDOWS]

    def cnt_of(slot):
        return block[slot, nseg * MAX_WINDOWS:].view(torch.int32).reshape(-1)[:nseg]

    def step(i, slot):
        rx.decode_capture(caps[i % len(caps)], seg_dev, MAX_WINDOWS, res_of(slot), cnt_of(slot), stream)

    def gather():
        if world > 1:
            dist.all_gather_into_tensor(g_block, block)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    for i in range(args.warmup):
        step(i, i % nslots)
    gather()
    barrier()

    def check(slot, cap_index):
        """correctness gate: records of one step against the generator's ground truth"""
        recs, cnt = capi.results_to_numpy(res_of(slot), cnt_of(slot), MAX_WINDOWS)
        truth = truths[cap_index]
        single = np.asarray(truth.get("n_replies", np.ones(nseg, dtype=np.int64))) == 1 if "n_replies" in truth else np.ones(nseg, bool)
        epc_ok = int((recs[:, 1]["crc_ok"] == 1).sum())
        rn_ok = int((recs[:, 0]["tag_id"] == np.asarray(truth["rn16"]))[single].sum())
        epc_match = int((recs[:, 1]["bits"] == np.asarray(truth["epc"])).all(axis=1)[single].sum())
        return {"epc_crc_ok": epc_ok, "rn16_match_truth": rn_ok, "epc_match_truth": epc_match, "segments": nseg,
                "single_reply_segments": int(single.sum()), "windows": int(cnt.sum())}

    gate0 = check((args.warmup - 1) % nslots, (args.warmup - 1) % len(caps))
    if fixed_q == 0:
        assert gate0["epc_crc_ok"] == nseg and gate0["epc_match_truth"] == nseg, "warm-up step decoded wrongly: %r" % (gate0,)
    block.zero_()           # a timed step that silently wrote nothing must not pass on warm-up records

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    rx.enable_kernel_timing(True)
    rx.kernel_time(reset=True)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t_host0 = time.perf_counter()
    ev0.record(stream)
    for i in range(args.steps):
        step(args.warmup + i, i % nslots)
        launches += rx.last_launch_count()
    gather()
    ev1.record(stream)
    barrier()
    t_host1 = time.perf_counter()
    ms = ev0.elapsed_time(ev1)
    k_ms, k_n = rx.kernel_time(reset=True)
    rx.enable_kernel_timing(False)
    clocks = None
    if rank == 0:
        sampler.stop()
        clocks = sampler.window(t_host0, t_host1)
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    total_raw = n_raw * world if cfg["scaling"] == "weak" else float(cfg["rounds"]) * slots * seg_len
    value = args.steps * total_raw / (ms_max * 1e-3) / 1e6
    last = args.steps - 1
    gate1 = check(last % nslots, (args.warmup + last) % len(caps))
    if fixed_q == 0:
        assert gate1["epc_crc_ok"] == nseg and gate1["epc_match_truth"] == nseg, "timed step decoded wrongly: %r" % (gate1,)
    if args.dump_outputs and rank == 0:
        # the records every rank holds after the closing all-gather, rank by rank
        parts = [capi.results_to_numpy(b[last % nslots, : nseg * MAX_WINDOWS],
                                       b[last % nslots, nseg * MAX_WINDOWS:].view(torch.int32).reshape(-1)[:nseg], MAX_WINDOWS)
                 for b in (g_block.unbind(0) if world > 1 else (block,))]
        dump_outputs(args.dump_outputs, np.concatenate([p[0] for p in parts]), np.concatenate([p[1] for p in parts]))

    # ------------------------------------------------------------------ sampled bit-exact parity against the oracle
    oracle_par = None
    if rank == 0:
        from oracle.pyoracle import Oracle
        stride = max(1, nseg // 256)
        pick = np.arange(0, nseg, stride)[:256]
        ci = (args.warmup + last) % len(caps)
        iq_pick = torch.cat([caps[ci][int(segs_np["offset"][s]): int(segs_np["offset"][s]) + seg_len] for s in pick]).cpu().numpy()
        segs_pick = abi.make_segments(np.arange(pick.size, dtype=np.uint64) * seg_len, [seg_len] * pick.size)
        orecs, ocnt, _ = Oracle(fixed_q=fixed_q, adc_rate=adc_rate, ntaps=ntaps).decode_segments(iq_pick, segs_pick, max_per_seg=MAX_WINDOWS)
        recs, cnt = capi.results_to_numpy(res_of(last % nslots), cnt_of(last % nslots), MAX_WINDOWS)
        mine = recs[pick].copy()
        mine["segment"] = np.arange(pick.size, dtype=np.int32)[:, None]
        exact = int(sum(mine[k].tobytes() == orecs[k].tobytes() and cnt[pick[k]] == ocnt[k] for k in range(pick.size)))
        oracle_par = {"sampled_segments": int(pick.size), "stride": int(stride), "bit_exact_vs_oracle": exact}
        assert exact == pick.size, "records differ from the oracle on sampled segments: %r" % (oracle_par,)

    # ------------------------------------------------------------------ end-to-end: host buffers through the C-ABI
    e2e_seg = min(nseg, 8000)
    e2e_raw = e2e_seg * seg_len
    h_iq = [torch.empty(e2e_raw, dtype=torch.complex64).pin_memory() for _ in range(2)]
    for b in range(2):
        h_iq[b].copy_(caps[b % len(caps)][:e2e_raw])
    h_res = torch.zeros((e2e_seg * MAX_WINDOWS, 64), dtype=torch.uint8).pin_memory()
    h_cnt = torch.zeros(e2e_seg, dtype=torch.int32).pin_memory()
    h_segs = torch.from_numpy(np.ascontiguousarray(segs_np[:e2e_seg]).view(np.uint8).copy()).pin_memory()
    e2e_steps = max(3, min(args.steps, 10))

    def e2e_step(i):
        rx.decode_capture_host_ptr(h_iq[i % 2].data_ptr(), e2e_raw, h_segs.data_ptr(), e2e_seg, MAX_WINDOWS,
                                   h_res.data_ptr(), h_cnt.data_ptr())

    for i in range(2):
        e2e_step(i)
    barrier()
    t0 = time.perf_counter()
    for i in range(e2e_steps):
        e2e_step(i)
    barrier()
    e2e_s = time.perf_counter() - t0
    te = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = e2e_steps * e2e_raw * world / float(te.item()) / 1e6
    e2e_recs = h_res.numpy().reshape(-1).view(abi.RESULT_DTYPE).reshape(e2e_seg, MAX_WINDOWS)
    e2e_ok = int((e2e_recs[:, 1]["crc_ok"] == 1).sum())

    if rank == 0:
        peak, peak_kind = hbm_peak()
        k_avg_ms = k_ms / max(1, k_n)
        achieved = 8.0 * n_raw / (k_avg_ms * 1e-3) / 1e9 if k_n else None
        traffic, traffic_src = None, None
        tp = os.path.join(ROOT, "profiles", "traffic.json")   # dram bytes per launch from the committed ncu --set full capture
        if os.path.exists(tp):
            try:
                tj = json.load(open(tp))
                if tj.get("segments") == nseg and tj.get("config", "cfg2") == args.config:
                    traffic = tj["dram_bytes_read"] + tj["dram_bytes_write"]
                    traffic_src = "profiles/traffic.json <- %s (ncu --set full of this kernel at this size; not measured in this run)" % tj.get("report", "?")
            except Exception:
                pass
        roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                    "frac": (achieved / peak) if achieved else None, "traffic": traffic, "traffic_source": traffic_src,
                    "kernel": kernel_name(adc_rate, ntaps),
                    "kernel_ms": k_avg_ms, "kernel_launches_timed": k_n, "peak_kind": peak_kind,
                    "algorithmic_bytes_per_launch": 8.0 * n_raw}
        cpu_b = None
        os.sched_setaffinity(0, affinity0)   # the CPU arm gets every usable core again, not just the GPU's NUMA node
        if not args.no_cpu_baseline:
            n_samp = min(nseg, 1000 if fixed_q == 0 else 2048)
            cap_cpu = synth.make_capture(n_samp, seed=1234, device="cpu", fixed_q=fixed_q, n_tags=n_tags, adc_rate=adc_rate)
            # bounded sample: ~10-30 s of CPU work = 6 x 40 passes over the sample, all usable CPUs
            r = cpu_reference_run(cap_cpu["iq"].numpy(), cap_cpu["segments"], steps=5, warmup=1, passes_per_step=40, fixed_q=fixed_q,
                                  adc_rate=adc_rate, ntaps=ntaps, what="%s sample" % args.config)
            cpu_b = {"value": r["value"], "unit": "MSamples/s", "cores": r["cores"], "kind": r["kind"], "sample": r["sample"]}
        line = {"metric": METRIC, "value": value, "unit": "MSamples/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": cfg["scaling"],
                "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config, "clocks": clocks,
                "e2e": {"value": e2e_value, "unit": "MSamples/s", "h2d_bytes_per_step": int(e2e_raw * 8 + h_segs.numel()),
                        "d2h_bytes_per_step": int(h_res.numel() + h_cnt.numel() * 4), "steps": e2e_steps,
                        "segments_per_step": e2e_seg, "epc_crc_ok": e2e_ok, "numa": numa},
                "gpu_launches": launches, "roofline": roofline, "cpu_baseline": cpu_b,
                "parity": {"warmup_step": gate0, "timed_step": gate1, "oracle": oracle_par}}
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def ingest(args, rank, local_rank):
    """SURVEY 8(f)-2 as a measured path: a recorded capture in HOST memory (the on-disk format of misc/data/file_source_test,
    apps/reader.py:102) -> rfid_b200_ingest_capture_host (sliced upload with the CW-gap segmenter's threshold pass behind
    every slice, segment table, decode) -> host records.  One GPU."""
    if rank != 0:
        return 0
    import torch
    from gen2_uhf_rfid_reader_b200 import abi, capi, synth
    assert torch.cuda.is_available(), "bench.py needs a GPU (there is no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    rounds = args.rounds or 1000
    rx = capi.Gen2Rx(device=local_rank)
    cap = synth.make_capture(rounds, seed=1234, device=dev)
    n_raw = cap["iq"].numel()
    rows = []
    for kind in ("pinned", "pageable"):
        h = torch.empty(n_raw, dtype=torch.complex64)
        if kind == "pinned":
            h = h.pin_memory()
        h.copy_(cap["iq"])
        iq_np = h.numpy()
        for _ in range(2):
            segs, recs, counts = rx.ingest_capture_host(iq_np, max_windows=MAX_WINDOWS)
        torch.cuda.synchronize(dev)
        ts = []
        for _ in range(args.steps):
            t0 = time.perf_counter()
            segs, recs, counts = rx.ingest_capture_host(iq_np, max_windows=MAX_WINDOWS)
            ts.append(time.perf_counter() - t0)
        t = float(np.median(ts))
        if args.dump_outputs and kind == "pinned":
            dump_outputs(args.dump_outputs, recs, counts,
                         extra={"segments_offset": segs["offset"], "segments_length": segs["length"]})
        ok = int(sum((recs[s, k]["crc_ok"] == 1) for s in range(len(segs)) for k in range(min(int(counts[s]), MAX_WINDOWS)) if recs[s, k]["kind"] == 1))
        rows.append({"host_memory": kind, "seconds_per_call": t, "msamples_per_s": n_raw / t / 1e6, "host_to_device_gbs": 8.0 * n_raw / t / 1e9,
                     "segments_found": int(len(segs)), "epc_crc_ok": ok, "launches_per_call": rx.last_launch_count()})
    line = {"metric": METRIC, "value": rows[0]["msamples_per_s"], "unit": "MSamples/s", "n_gpus": 1, "steps": args.steps, "warmup": 2,
            "ms_per_step": rows[0]["seconds_per_call"] * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": {"workload": "ingest: %d-round capture (%.1f MB) in host memory -> segmenter + decode -> host records; wall clock per call, "
                                   "host<->device copies inside" % (rounds, n_raw * 8 / 1e6), "config": "ingest",
                       "hbm_bytes_per_sample": "16 algorithmic (the threshold pass and the decode each read the capture once) + 8 written by the upload"},
            "e2e": {"value": rows[0]["msamples_per_s"], "unit": "MSamples/s", "h2d_bytes_per_step": int(n_raw * 8), "d2h_bytes_per_step": int(rounds * MAX_WINDOWS * 64)},
            "ingest": rows, "gpu_launches": rows[0]["launches_per_call"] * args.steps}
    print(json.dumps(line))
    return 0


def sweep(args, rank, local_rank, world):
    """cfg5: kernel GB/s against the HBM roofline at raw rates 1 .. 8 MS/s (one GPU; other ranks idle)."""
    if rank != 0:
        return 0
    import torch
    from gen2_uhf_rfid_reader_b200 import abi, capi, synth
    from oracle.pyoracle import Oracle
    assert torch.cuda.is_available(), "bench.py needs a GPU (there is no CPU fallback)"
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(local_rank)
    rounds = args.rounds or 1000
    peak, peak_kind = hbm_peak()
    rows = []
    for adc in SWEEP_RATES:
        ntaps = ntaps_for(adc)
        rx = capi.Gen2Rx(device=local_rank, adc_rate=adc, ntaps=ntaps)
        caps = [synth.make_capture(rounds, seed=1234 + 17 * b, device=dev, adc_rate=adc) for b in range(2)]
        segs_np = caps[0]["segments"]
        seg_dev = capi.segments_to_device(segs_np, dev)
        n_raw = caps[0]["iq"].numel()
        res = torch.zeros((rounds * MAX_WINDOWS, 64), dtype=torch.uint8, device=dev)
        cnt = torch.zeros(rounds, dtype=torch.int32, device=dev)
        for i in range(args.warmup):
            rx.decode_capture(caps[i % 2]["iq"], seg_dev, MAX_WINDOWS, res, cnt)
        torch.cuda.synchronize(dev)
        rx.enable_kernel_timing(True)
        rx.kernel_time(reset=True)
        for i in range(args.steps):
            rx.decode_capture(caps[(args.warmup + i) % 2]["iq"], seg_dev, MAX_WINDOWS, res, cnt)
        torch.cuda.synchronize(dev)
        k_ms, k_n = rx.kernel_time(reset=True)
        rx.enable_kernel_timing(False)
        recs, counts = capi.results_to_numpy(res, cnt, MAX_WINDOWS)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, recs, counts, prefix="adc%d_" % adc, limit=DUMP_BYTES // len(SWEEP_RATES))
        ci = (args.warmup + args.steps - 1) % 2
        # parity on a sample of the segments against the oracle at this rate
        pick = np.arange(0, rounds, max(1, rounds // 64))[:64]
        seg_len = int(segs_np["length"][0])
        iq_pick = torch.cat([caps[ci]["iq"][int(segs_np["offset"][s]): int(segs_np["offset"][s]) + seg_len] for s in pick]).cpu().numpy()
        segs_pick = abi.make_segments(np.arange(pick.size, dtype=np.uint64) * seg_len, [seg_len] * pick.size)
        orecs, ocnt, _ = Oracle(adc_rate=adc, ntaps=ntaps).decode_segments(iq_pick, segs_pick, max_per_seg=MAX_WINDOWS)
        mine = recs[pick].copy()
        mine["segment"] = np.arange(pick.size, dtype=np.int32)[:, None]
        exact = int(sum(mine[k].tobytes() == orecs[k].tobytes() and counts[pick[k]] == ocnt[k] for k in range(pick.size)))
        k_avg = k_ms / max(1, k_n)
        gbs = 8.0 * n_raw / (k_avg * 1e-3) / 1e9
        rows.append({"adc_rate": adc, "fs_dec": adc // 5, "ntaps": ntaps, "ntaps_note": "12.5 rounded to 12" if adc == 1_000_000 else None,
                     "kernel": kernel_name(adc, ntaps), "segments": rounds, "segment_samples": seg_len, "kernel_us": 1e3 * k_avg,
                     "achieved_gbs": gbs, "frac": gbs / peak, "msamples_per_s": n_raw / (k_avg * 1e-3) / 1e6,
                     "epc_crc_ok": int((recs[:, 1]["crc_ok"] == 1).sum()), "oracle_sampled": int(pick.size), "oracle_bit_exact": exact})
        del rx, caps
        torch.cuda.empty_cache()
    ref = [r for r in rows if r["adc_rate"] == 2_000_000][0]
    line = {"metric": METRIC, "value": ref["msamples_per_s"], "unit": "MSamples/s", "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ref["kernel_us"] / 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": {"workload": "cfg5: raw-rate sweep 1/2/4/6/8 MS/s, decimation 5, ntaps = rate/(2 BLF), %d inventory rounds of %.0f us per rate; "
                                   "value = the 2 MS/s row (kernel time only: this is a kernel-bandwidth sweep, no collective, no host copies)" % (rounds, SEG_US),
                       "config": "cfg5"},
            "roofline": {"bound": "hbm", "peak": peak, "peak_kind": peak_kind, "unit": "GB/s", "achieved": ref["achieved_gbs"], "frac": ref["frac"],
                         "traffic": None},
            "sweep": rows, "gpu_launches": args.steps * len(rows)}
    print(json.dumps(line))
    return 0


if __name__ == "__main__":
    sys.exit(main())
