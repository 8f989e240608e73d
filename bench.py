#!/usr/bin/env python
"""bench.py -- audio Msamples/s demodulated over batched streams (BASELINE.json).

One "step" = one pass of the hot path (the batched rx loop: per-stream frame
search + tone correlation + rx state machine, src/minimodem.c:1137-1463 over
src/fsk.c:449-538) over one batch of synthetic streams.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

N>1 is launched by torchrun (one rank per GPU); streams shard across ranks with
no data-path collective (weak scaling: every rank demodulates its own batch);
NCCL carries only the broadcast of the derived plan (fsk_b200_rx_params) and the
all-reduce of the timing / frame-count scalars.

`value`   : whole-job Msamples/s of the HEADLINE workload (BASELINE configs[1]: 1200 baud,
            48 kHz, 65 536 streams per GPU), inputs resident in HBM, timed with CUDA events.
`e2e`     : the same metric through the host-buffer C-ABI call
            (fsk_b200_rx_batch_host): pinned host samples -> device -> records
            back on the host, copies inside the timed region.
`roofline`: algorithmic bytes (4 + 20/frame_nsamples per sample, SURVEY.md 8d)
            over the rx kernel's own CUDA-event time, against the measured HBM
            copy bandwidth (MEASURED_PEAKS.json).
`configs` : the other BASELINE configurations (RTTY 45.45 @8 kHz, Bell103 300 baud with the
            reference's -f offset sweep and with AWGN, NOAA SAME per-GPU shard) and a noisy
            variant of the headline, each with its own value / kernel_ms / roofline fraction /
            candidates per frame counted on the device / decode check on >= 1 % of the streams.
`cpu_baseline` / `--impl reference`: the reference's CPU implementation (the
            unmodified src/fsk.c compiled into oracle/_ref behind the oracle's
            rx-loop restatement; else the oracle port) on the host cores, on a
            bounded sample of the same workload, run by a persistent pinned worker pool.
"""
import argparse
import ctypes as C
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True          # no __pycache__ in the tree: it may be read-only
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402

METRIC = "audio Msamples/s demodulated (batched streams)"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--mode", default=os.environ.get("FSK_BENCH_MODE", "1200"))
    ap.add_argument("--rate", type=int, default=int(os.environ.get("FSK_BENCH_RATE", "48000")))
    ap.add_argument("--streams", type=int, default=int(os.environ.get("FSK_BENCH_STREAMS", "65536")),
                    help="streams per GPU")
    ap.add_argument("--nsamples", type=int, default=int(os.environ.get("FSK_BENCH_NSAMPLES", "192000")),
                    help="samples per stream (4 s at 48 kHz)")
    ap.add_argument("--amplitude", type=float, default=1.0)
    ap.add_argument("--awgn", type=float, default=0.0, help="sigma of additive white gaussian noise on the headline")
    ap.add_argument("--offset", type=float, default=0.0, help="constant offset -f (the reference's --Xrxnoise)")
    ap.add_argument("--e2e-streams", type=int, default=0, help="0 = the whole batch at N=1, 16384 per rank otherwise")
    ap.add_argument("--cpu-streams", type=int, default=0, help="CPU sample size (0 = 64 per core, at most 8192)")
    ap.add_argument("--config-steps", type=int, default=3, help="timed steps for each entry of `configs`")
    ap.add_argument("--lanes", type=int, default=0)
    ap.add_argument("--wpb", type=int, default=0)
    ap.add_argument("--ring", type=int, default=0)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-configs", action="store_true")
    ap.add_argument("--only-config", default="", help="run only the `configs` entries whose key contains this")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write the frame records and stream states of the headline's last timed step to DIR/*.npy")
    return ap.parse_args()


def workload_name(mode, rate, S, n, extra=""):
    return "%s baud, %d Hz float32, %d synthetic streams x %d samples per GPU%s" % (mode, rate, S, n, extra)


# --------------------------------------------------------------------------
# CPU arm (the reference on the host cores)
# --------------------------------------------------------------------------
def cpu_streams_on_host(mode_name, rate, nsamples, ndistinct):
    """Synthetic streams for the CPU arm, made on the CPU by the oracle's TX
    restatement (same signal model and payload statistics as the device generator)."""
    import orc
    m = orc.Mode(mode_name, sample_rate=rate)
    d = m.derived()
    one = int(orc.lib().orc_tx_nsamples(C.byref(m.tx_config(1.0, 4096, True)), 1))
    zero = int(orc.lib().orc_tx_nsamples(C.byref(m.tx_config(1.0, 4096, True)), 2)) - one
    nwords = max(1, (nsamples - (one - zero) - int(d.nsamples_per_bit)) // zero)
    rng = np.random.default_rng(20260922)
    x = np.zeros((ndistinct, nsamples), np.float32)
    for s in range(ndistinct):
        words = rng.integers(32, 127, nwords, dtype=np.uint32) & ((1 << m.n_data_bits) - 1)
        w = orc.tx_words(m, words, 1.0, 4096, True)
        lead = 0 if m.do_rx_sync else int(rng.integers(0, max(1, int(d.nsamples_per_bit))))
        k = min(w.size, nsamples - lead)
        x[s, lead:lead + k] = w[:k]
    return m, x


def cpu_measure(mode, x, nsamples, nstreams, steps, warmup, want_port=False):
    """Times the CPU arm: `nstreams` streams (the rows of `x`, repeated as often as needed -- every
    copy is its own memory) through a persistent pool of pinned workers (orc.RxPool: one plan per
    worker built once, contiguous stream blocks first-touched by their worker).  The thread count is
    chosen by one untimed pass each at all / half of the allowed CPUs; then `warmup` untimed and
    `steps` timed passes.  `value` is the FASTEST pass, `median` the median one: on the shared hosts of the pool a
    pass of the same work lands either at ~0.30 s or at ~0.39 s, so a median of three or five flips between the two
    (4.1-5.1 Gsamples/s from run to run) while the minimum reproduces within 2 % -- and it is the conservative
    choice for every speed-up quoted against this arm.

    kind "reference" = the unmodified src/fsk.c.  Its speed is its FFT library's: it is timed on
    MKL's DFTI (oracle/_ref/libfsk_ref_dfti.so, the closest thing to FFTW in this image; not
    FFTW) when that loads, else on the portable scalar FFT stand-in, and `sample` says which."""
    import orc
    cores = len(os.sched_getaffinity(0))
    kind = "reference" if orc.have_ref() else "port"
    impl = {"port": "port", "reference": "reference"}
    fft = "portable scalar mixed-radix FFT stand-in (not FFTW)"
    if orc.have_ref() and orc.have_ref_dfti():
        try:
            orc.rx_many(mode, x[:1], nsamples=nsamples, nthreads=1, kind="reference-dfti")   # MKL start-up
            impl["reference"] = "reference-dfti"
            fft = "MKL DFTI FFT from libtorch_cpu.so as the FFTW stand-in (not FFTW)"
        except Exception:
            pass
    reps = (nstreams + x.shape[0] - 1) // x.shape[0]
    batch = np.tile(x, (reps, 1))[:nstreams] if reps > 1 else x[:nstreams]
    out = {}
    check = None
    for k in ([kind, "port"] if (want_port and kind != "port") else [kind]):
        cands = []
        for nt in sorted({cores, max(1, cores // 2)}, reverse=True):
            pool = orc.RxPool(mode, nt, impl[k])
            pool.load(batch, nsamples)
            dt, _, _, _ = pool.run()                       # untimed: picks the thread count
            cands.append((dt, nt, pool))
        cands.sort(key=lambda c: c[0])
        for c in cands[1:]:
            c[2].close()
        _, nt, pool = cands[0]
        ts = []
        total = bx = None
        for i in range(warmup + steps):
            dt, total, _, bx = pool.run()
            if i >= warmup:
                ts.append(dt)
        pool.close()
        sig = (int(total), int(np.bitwise_xor.reduce(bx)))
        if check is None:
            check = sig
        med, best = float(np.median(ts)), float(min(ts))
        nsam = nstreams * nsamples
        out[k] = dict(value=nsam / best / 1e6, best=nsam / best / 1e6, median=nsam / med / 1e6, unit="Msamples/s",
                      cores=nt, kind=k, passes=len(ts), seconds_per_pass=best, seconds_median_pass=med, seconds_best_pass=best,
                      seconds_all_passes=[round(t, 4) for t in ts],
                      sample="%d streams x %d samples per pass (%d distinct streams, each copy its own memory); "
                             "persistent pool of %d pinned threads (best of {%d, %d}), plans built once outside the "
                             "timed passes, contiguous per-thread stream blocks first-touched by their thread; "
                             "value = fastest of %d passes (median reported beside it); %s" % (
                                 nstreams, nsamples, x.shape[0], nt, cores, max(1, cores // 2), len(ts),
                                 "unmodified src/fsk.c (oracle/_ref) on the %s, behind the oracle rx loop" % fft
                                 if k == "reference" else "oracle port (two-bin direct DFT, no FFT): best-case CPU"),
                      frames=int(total), same_frames_as_first_arm=bool(sig == check))
    return out[kind], out


def cpu_sample_streams(a):
    cores = len(os.sched_getaffinity(0))
    return a.cpu_streams or max(16, min(8192, 64 * cores))


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n = cpu_sample_streams(a)
    mode, x = cpu_streams_on_host(a.mode, a.rate, a.nsamples, min(n, 128))
    cb, _ = cpu_measure(mode, x, a.nsamples, n, steps=max(1, a.steps), warmup=a.warmup)
    line = {
        "impl": "reference", "metric": METRIC,
        "value": cb["value"], "unit": "Msamples/s", "n_gpus": a.gpus, "steps": a.steps,
        "warmup": a.warmup, "ms_per_step": cb["seconds_per_pass"] * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(a.mode, a.rate, a.streams, a.nsamples),
                   "sample_per_step": cb["sample"]},
        "cpu_baseline": cb,
        "e2e": {"value": cb["value"], "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# --------------------------------------------------------------------------
# clocks
# --------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                       "--format=csv,noheader,nounits", "-lms", "100"],
                                      stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.p = None

    def _read(self):
        for ln in self.p.stdout:
            self.rows.append([c.strip() for c in ln.split(",")])

    def stop(self):
        if not self.p:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        try:
            self.p.wait(timeout=2)
        except Exception:
            self.p.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                for k, nm in enumerate(names):
                    if r[5 + k].lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# --------------------------------------------------------------------------
# GPU arm
# --------------------------------------------------------------------------
def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def _code_only(text):
    """C/CUDA source without comments and without white space (string and character literals kept as they are):
    what the compiler sees, so a comment edit does not cut an ncu figure loose from the build it was taken on."""
    out, i, n = [], 0, len(text)
    while i < n:
        c = text[i]
        if c == "/" and i + 1 < n and text[i + 1] == "*":
            j = text.find("*/", i + 2)
            i = n if j < 0 else j + 2
            out.append(" ")
        elif c == "/" and i + 1 < n and text[i + 1] == "/":
            j = text.find("\n", i)
            i = n if j < 0 else j
        elif c in "\"'":
            j = i + 1
            while j < n and text[j] != c:
                j += 2 if text[j] == "\\" else 1
            out.append(text[i:j + 1])
            i = j + 1
        else:
            out.append(c)
            i += 1
    return " ".join("".join(out).split())


def kernel_source_hash():
    """sha256 over the CUDA sources of the rx kernel, comments and white space removed: ties an ncu DRAM-traffic
    figure to the build."""
    h = hashlib.sha256()
    for f in ("fsk_b200_kernels.cu", "fsk_b200_device.cuh", "fsk_b200_internal.h"):
        h.update(_code_only(open(os.path.join(ROOT, "minimodem_b200", "csrc", f), encoding="utf-8", errors="replace").read()).encode())
    return h.hexdigest()[:16]


def measured_traffic(mode, rate, S, n):
    """DRAM bytes per launch from the committed `ncu --set full` capture of this workload --
    only if that capture was taken on THIS kernel source (hash match); else None."""
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "r2_traffic.json")))
    except Exception:
        return None
    src = kernel_source_hash()
    for e in tj.get("captures", []):
        w = e["workload"]
        if e.get("kernel_source_sha16") == src and (w["mode"], w["rate"], w["streams"], w["nsamples"]) == (mode, rate, S, n):
            return e["dram_bytes_read"] + e["dram_bytes_write"]
    return None


class Workload:
    """Synthetic streams in the reference transmitter's signal model, generated on the device
    (fsk_b200_tx_batch, bit-exact with the oracle's TX restatement), plus optional additive noise."""

    def __init__(self, mm, torch, dev, rank, mode, rate, S, n, amplitude=1.0):
        self.mm, self.torch, self.dev = mm, torch, dev
        self.mode, self.rate, self.S, self.n = mode, rate, S, n
        self.cfg = mm.rx_config_for_mode(mode, rate)
        self.params = mm.rx_params(self.cfg)
        self.stride = (n + 3) & ~3
        cfg, params = self.cfg, self.params
        tcfg = mm.tx_config_from(cfg)
        spb = float(params.nsamples_per_bit)
        # transmitter frame length (src/minimodem.c:131-132, :96-111: size_t * float truncations)
        bit = int(np.float32(np.float32(int(cfg.sample_rate)) / np.float32(cfg.data_rate)) + np.float32(0.5))
        tx_frame = (int(np.float32(bit) * np.float32(tcfg.nstartbits)) if tcfg.nstartbits > 0 else 0) \
            + params.n_data_bits * bit + (int(np.float32(bit) * np.float32(tcfg.nstopbits)) if tcfg.nstopbits > 0 else 0)
        max_lead = 0 if cfg.do_rx_sync else max(1, int(spb))   # no lead-in for sync modes (see tests)
        overhead = (tcfg.leader_bits + tcfg.trailer_bits) * bit + tcfg.do_tx_sync_bytes * tx_frame + max_lead
        self.nwords = max(1, (n - overhead) // tx_frame)
        gen = torch.Generator(device="cpu").manual_seed(20260922 + rank)
        self.mask = (1 << params.n_data_bits) - 1
        lo, hi = (32, 127) if params.n_data_bits >= 7 else (0, 1 << params.n_data_bits)
        self.words = (torch.randint(lo, hi, (S, self.nwords), generator=gen, dtype=torch.int32) & self.mask).to(dev)
        lead = (torch.randint(0, max_lead, (S,), generator=gen, dtype=torch.int32) if max_lead
                else torch.zeros(S, dtype=torch.int32)).to(dev)
        table = torch.from_numpy(mm.sin_table(4096, amplitude)).to(dev)
        self.x = torch.empty((S, self.stride), dtype=torch.float32, device=dev)
        mm.tx_batch(tcfg, self.words, n, lead_in=lead, table=table, out=self.x, stride=self.stride)
        torch.cuda.synchronize()
        self.shift = (1 if params.nstopbits != 0 else 0) + params.nstartbits

    def perturbed(self, awgn=0.0, offset=0.0, seed=1):
        """x + N(0, awgn^2) - offset into a new buffer (chunked so the temporaries stay small)."""
        torch = self.torch
        y = torch.empty_like(self.x)
        g = torch.Generator(device=self.dev).manual_seed(seed)
        rows = max(1, (256 << 20) // (self.stride * 4))
        for s0 in range(0, self.S, rows):
            blk = self.x[s0:s0 + rows]
            if awgn:
                y[s0:s0 + rows] = blk + awgn * torch.randn(blk.shape, generator=g, device=self.dev, dtype=torch.float32)
            else:
                y[s0:s0 + rows] = blk
            if offset:
                y[s0:s0 + rows] -= offset            # src/simpleaudio-sndfile.c:64-70: the reference's --Xrxnoise
        torch.cuda.synchronize()
        return y

    def decode_check(self, frames, states, sample_rows):
        """Decoded data words of the sampled streams against what was transmitted.  Returns the
        fraction of sampled streams whose whole payload appears, in order, in the decoded words."""
        mm = self.mm
        st = mm.states_to_numpy(states[sample_rows])
        fr = mm.frames_to_numpy(frames[sample_rows])
        w = self.words[sample_rows].cpu().numpy() & self.mask
        ok = 0
        for i in range(len(st)):
            recs = fr[i, :st["nframes"][i]]
            recs = recs[recs["frame_start"] != mm.FRAME_REPORT]
            data = (recs["bits_lo"].astype(np.int64) >> self.shift) & self.mask
            if self.cfg.do_rx_sync:
                data = data[data != (self.cfg.sync_byte & self.mask)]      # the rx drops sync bytes (:1436-1439)
            want = w[i]
            L = len(want)
            hit = False
            for k in range(0, max(1, len(data) - L + 1)):
                if len(data) - k >= L and np.array_equal(data[k:k + L], want):
                    hit = True
                    break
            ok += hit
        return ok / max(1, len(st))


def time_rx(torch, dist, world, dev, eng, x, n, max_frames, frames, states, steps, warmup, sampler=None):
    """`warmup` untimed + `steps` timed passes of the rx kernel over x; CUDA events on the launching
    stream (torch's current stream, which is where eng.rx_batch launches).  Returns (ms_per_step, kernel_ms)."""
    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(warmup):
        states.zero_()
        eng.rx_batch(x, nsamples=n, max_frames=max_frames, frames=frames, states=states)
    barrier()
    if sampler:
        sampler.start()
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t0.record()
    for i in range(steps):
        states.zero_()
        kev[i][0].record()
        eng.rx_batch(x, nsamples=n, max_frames=max_frames, frames=frames, states=states)
        kev[i][1].record()
    t1.record()
    barrier()
    clocks = sampler.stop() if sampler else None
    ms_kernel = sum(e0.elapsed_time(e1) for e0, e1 in kev) / steps
    ms_step = t0.elapsed_time(t1) / steps
    if world > 1:
        t = torch.tensor([ms_step, ms_kernel], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_step, ms_kernel = float(t[0]), float(t[1])
    return ms_step, ms_kernel, clocks


def dump_outputs(mm, torch, out_dir, frames, states, budget=60_000_000):
    """What rx_batch handed its caller in the last timed step, as float64 arrays (exact for every field):
    DIR/frames_<field>.npy [k, max_frames] per frame-record field, zero past each stream's nframes (those
    slots hold no record), DIR/states_<field>.npy [k] per stream-state field, and DIR/streams.npy, the
    rows they belong to -- all streams, or a fixed seeded sample of them that keeps the files under `budget`."""
    S, max_frames = frames.shape[0], frames.shape[1]
    per_stream = 8 * (1 + max_frames * len(mm.FRAME_DTYPE.names) + len(mm.STATE_DTYPE.names))
    k = min(S, max(1, budget // per_stream))
    rows = np.arange(S) if k == S else np.sort(np.random.default_rng(20260922).choice(S, k, replace=False))
    sel = torch.from_numpy(rows).to(frames.device)
    fr = mm.frames_to_numpy(frames.index_select(0, sel))
    st = mm.states_to_numpy(states.index_select(0, sel))
    valid = np.arange(max_frames)[None, :] < st["nframes"].astype(np.int64)[:, None]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "streams.npy"), rows.astype(np.float64))
    for f in mm.FRAME_DTYPE.names:
        np.save(os.path.join(out_dir, "frames_%s.npy" % f), np.where(valid, fr[f], 0).astype(np.float64))
    for f in mm.STATE_DTYPE.names:
        np.save(os.path.join(out_dir, "states_%s.npy" % f), st[f].astype(np.float64))


def summarize(mm, torch, dist, world, dev, wl, frames, states, ms_step, ms_kernel, clean, peak):
    """Per-workload result block: throughput, roofline fraction, device-side statistics, decode check."""
    S, n = wl.S, wl.n
    st = mm.states_to_numpy(states)
    assert (st["done"] == 1).all(), "streams did not finish"
    nfr = st["nframes"].astype(np.int64)
    ncand = st["stat_candidates"].astype(np.int64)
    nsrch = st["stat_searches"].astype(np.int64)
    nrows = max(8, (S + 99) // 100)                                  # >= 1 % of the streams
    rows = torch.arange(0, S, max(1, S // nrows), device=dev)[:nrows]
    okfrac = wl.decode_check(frames, states, rows)
    if clean:
        assert nfr.min() >= wl.nwords, ("frames per stream", int(nfr.min()), wl.nwords)
        assert okfrac == 1.0, ("decode mismatch on clean streams", okfrac)
    tot = torch.tensor([float(nfr.sum()), float(ncand.sum()), float(nsrch.sum()),
                        float(np.bitwise_xor.reduce(mm.frames_to_numpy(frames[rows])["bits_lo"].reshape(-1)) & 0xFFFFFF)],
                       dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    frames_total, cand_total, srch_total = float(tot[0]), float(tot[1]), float(tot[2])
    bps = 4.0 + 20.0 / wl.params.frame_nsamples
    achieved = S * n * bps / (ms_kernel * 1e-3) / 1e9
    return {
        "value": S * n * world / (ms_step * 1e-3) / 1e6, "unit": "Msamples/s",
        "ms_per_step": ms_step, "kernel_ms": ms_kernel,
        "streams_per_gpu": S, "nsamples": n, "frame_nsamples": wl.params.frame_nsamples,
        "roofline_frac": achieved / peak, "achieved_gbs": achieved, "algorithmic_bytes_per_sample": bps,
        "frames_decoded": int(frames_total),
        "candidates_per_frame": cand_total / max(1.0, frames_total),
        "candidates_per_search": cand_total / max(1.0, srch_total),
        "searches_per_frame": srch_total / max(1.0, frames_total),
        "decode_check": {"streams": int(len(rows)), "fraction_exact": okfrac},
    }


def run_ours(a):
    import torch
    import torch.distributed as dist
    import minimodem_b200 as mm

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "").upper() not in ("INFO", "TRACE"):
            os.environ["NCCL_DEBUG"] = "ERROR"      # keep stdout to the one JSON line
        dist.init_process_group("nccl", device_id=dev)
    peak, peak_src = peaks()

    def engine_for(wl):
        # plan: derived on rank 0, broadcast over NCCL (the only collective on the data path)
        params = wl.params
        if world > 1:
            from minimodem_b200 import dist as mdist
            params = mdist.broadcast_params(params if rank == 0 else None, src=0, device=dev)
        eng = mm.RxEngine(params)
        if a.lanes or a.wpb or a.ring:
            eng.tune(a.lanes, a.wpb, a.ring)
        return eng

    # ---- headline workload
    S, n = a.streams, a.nsamples
    free, _ = torch.cuda.mem_get_info(dev)
    stride = (n + 3) & ~3
    shrunk = False
    while S * stride * 4 * (2 if (a.awgn or a.offset) else 1) > 0.80 * free and S > 1024:
        S //= 2
        shrunk = True
    wl = Workload(mm, torch, dev, rank, a.mode, a.rate, S, n, a.amplitude)
    x = wl.perturbed(a.awgn, a.offset) if (a.awgn or a.offset) else wl.x
    eng = engine_for(wl)
    max_frames = eng.max_frames(n)
    frames = torch.empty((S, max_frames, 5), dtype=torch.int32, device=dev)
    states = torch.zeros((S, mm.STATE_WORDS), dtype=torch.int32, device=dev)
    launches0 = mm.launch_count()
    sampler = ClockSampler(local) if rank == 0 else None
    ms_step, ms_kernel, clocks = time_rx(torch, dist, world, dev, eng, x, n, max_frames, frames, states,
                                         a.steps, a.warmup, sampler)
    launches = mm.launch_count() - launches0 - a.warmup
    if a.dump_outputs and rank == 0:
        dump_outputs(mm, torch, a.dump_outputs, frames, states)
    head = summarize(mm, torch, dist, world, dev, wl, frames, states, ms_step, ms_kernel,
                     clean=not (a.awgn or a.offset), peak=peak)
    st = mm.states_to_numpy(states)
    value = head["value"]
    frame = wl.params.frame_nsamples
    bytes_per_sample = head["algorithmic_bytes_per_sample"]
    roofline = {"bound": "hbm", "achieved": head["achieved_gbs"], "peak": peak, "unit": "GB/s",
                "frac": head["roofline_frac"], "traffic": measured_traffic(a.mode, a.rate, S, n),
                "algorithmic_bytes": S * n * bytes_per_sample, "peak_source": peak_src, "kernel": "k_rx",
                "kernel_variant": eng.last_kernel(),
                "kernel_ms": ms_kernel, "algorithmic_bytes_per_sample": bytes_per_sample,
                "kernel_source_sha16": kernel_source_hash(),
                "candidates_per_frame": head["candidates_per_frame"],
                "decode_check": head["decode_check"],
                "confidence_note": "fast path: sqrt.approx/div.approx + tree-ordered sums; confidence within "
                                   "~1e-6 relative of the reference (tested to 1e-4), bits/frame positions exact"}

    # ---- end to end through the host-buffer C ABI call
    e2e = None
    if not a.no_e2e:
        E = min(a.e2e_streams or (S if world == 1 else 16384), S)
        hx = torch.empty((E, stride), dtype=torch.float32, pin_memory=True)
        hx.copy_(x[:E])
        hfr = torch.empty((E, max_frames, 5), dtype=torch.int32, pin_memory=True)
        hst = torch.zeros((E, mm.STATE_WORDS), dtype=torch.int32, pin_memory=True)
        torch.cuda.synchronize()
        launches_e0 = mm.launch_count()

        def timed_host(fn, steps, warm):
            for _ in range(warm):
                hst.zero_()
                fn()
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            ts = []
            for _ in range(steps):
                hst.zero_()
                tt = time.perf_counter()
                fn()
                ts.append(time.perf_counter() - tt)
            dt = sum(ts) / len(ts)
            if world > 1:
                t = torch.tensor([dt], dtype=torch.float64, device=dev)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                dt = float(t[0])
            return dt

        esteps = max(2, min(a.steps, 3))
        dt = timed_host(lambda: eng.rx_batch_host(hx, nsamples=n, max_frames=max_frames, frames_out=hfr,
                                                  states_out=hst), esteps, 1)
        hs = hst.numpy().view(mm.STATE_DTYPE).reshape(-1)
        assert (hs["done"] == 1).all() and np.array_equal(hs["nframes"], st["nframes"][:E])
        # N2: the same streams as 16-bit PCM, 2 bytes per sample on PCIe and in HBM
        hx16 = torch.empty((E, stride), dtype=torch.int16, pin_memory=True)
        rows = max(1, (256 << 20) // (stride * 4))
        for s0 in range(0, E, rows):
            hx16[s0:s0 + rows].copy_((x[s0:min(E, s0 + rows)] * 32767.0).round().clamp_(-32768, 32767).to(torch.int16))
        torch.cuda.synchronize()
        dt16 = timed_host(lambda: eng.rx_batch_host_s16(hx16, nsamples=n, max_frames=max_frames, frames_out=hfr,
                                                        states_out=hst), esteps, 1)
        hs16 = hst.numpy().view(mm.STATE_DTYPE).reshape(-1)
        assert (hs16["done"] == 1).all() and (a.awgn or a.offset or int(hs16["nframes"].min()) >= wl.nwords)
        e2e = {"value": E * n * world / dt / 1e6, "unit": "Msamples/s",
               "h2d_bytes_per_step": int(E * stride * 4 + E * 4 * mm.STATE_WORDS),
               "d2h_bytes_per_step": int(E * max_frames * 20 + E * 4 * mm.STATE_WORDS),
               "streams_per_step": E, "ms_per_step": dt * 1e3, "h2d_gbs": E * stride * 4 / dt / 1e9,
               "launches": int(mm.launch_count() - launches_e0),
               "note": "fsk_b200_rx_batch_host on pinned host float32 buffers; PCIe-bound (4 B/sample in)",
               "s16_ingest": {"value": E * n * world / dt16 / 1e6, "unit": "Msamples/s", "ms_per_step": dt16 * 1e3,
                              "h2d_bytes_per_step": int(E * stride * 2 + E * 4 * mm.STATE_WORDS),
                              "h2d_gbs": E * stride * 2 / dt16 / 1e9,
                              "ratio_to_float": dt / dt16,
                              "note": "fsk_b200_rx_batch_host_s16: int16 PCM host streams (N2), widened inside the rx "
                                      "kernel's ring fill: 2 B/sample on PCIe and in HBM"}}
        del hx, hx16, hfr, hst

    # ---- the reference CPU path on this box's host cores (rank 0, N=1 only), on a sample of these streams
    cpu = None
    cpu_best = None
    if rank == 0 and world == 1 and not a.no_cpu:
        try:
            import orc
            ncpu = cpu_sample_streams(a)
            hostx = np.ascontiguousarray(x[:min(128, S), :n].cpu().numpy())
            cpu, both = cpu_measure(orc.Mode(a.mode, sample_rate=a.rate), hostx, n, ncpu, steps=5, warmup=1,
                                    want_port=True)
            cpu_best = both.get("port") if both.get("port") is not cpu else None
        except Exception as ex:  # the checker is optional for the number, never for the tests
            cpu = {"value": None, "unit": "Msamples/s", "cores": None, "kind": "unavailable", "sample": repr(ex)}

    # ---- the other BASELINE configurations
    configs = []
    if not a.no_configs:
        del frames, states
        if x is not wl.x:
            del x
        del wl
        torch.cuda.empty_cache()
        plan = [
            # key, mode, rate, streams, nsamples, amplitude, [(suffix, awgn, offset)]
            ("cfg2_1200_awgn", "1200", 48000, 65536, 192000, 1.0, [("0.35", 0.35, 0.0)]),
            ("cfg3_rtty_8k", "rtty", 8000, 262144, 32000, 1.0, [("clean", 0.0, 0.0)]),
            ("cfg4_bell103", "300", 48000, 32768, 192000, 0.5,
             [("offset0.00", 0.0, 0.0), ("offset0.05", 0.0, 0.05), ("offset0.10", 0.0, 0.10), ("offset0.50", 0.0, 0.50),
              ("awgn0.05", 0.05, 0.0), ("awgn0.10", 0.10, 0.0), ("awgn0.50", 0.50, 0.0)]),
            ("cfg5_same_per_gpu", "same", 48000, 131072, 24000, 1.0, [("clean", 0.0, 0.0)]),
        ]
        for key, mode, rate, cS, cn, amp, variants in plan:
            if a.only_config and a.only_config not in key:
                continue
            free, _ = torch.cuda.mem_get_info(dev)
            while cS * ((cn + 3) & ~3) * 4 * 2 > 0.85 * free and cS > 1024:
                cS //= 2
            cwl = Workload(mm, torch, dev, rank, mode, rate, cS, cn, amp)
            ceng = engine_for(cwl)
            cmax = ceng.max_frames(cn)
            cfr = torch.empty((cS, cmax, 5), dtype=torch.int32, device=dev)
            cst = torch.zeros((cS, mm.STATE_WORDS), dtype=torch.int32, device=dev)
            for suffix, awgn, offset in variants:
                cx = cwl.perturbed(awgn, offset) if (awgn or offset) else cwl.x
                ms_s, ms_k, _ = time_rx(torch, dist, world, dev, ceng, cx, cn, cmax, cfr, cst, a.config_steps, 3)
                r = summarize(mm, torch, dist, world, dev, cwl, cfr, cst, ms_s, ms_k,
                              clean=not (awgn or offset), peak=peak)
                r.update({"key": "%s_%s" % (key, suffix), "kernel": ceng.last_kernel(),
                          # DRAM bytes of one launch of this workload's clean variant, if profiles/ holds an ncu
                          # capture of it taken on this kernel source (else None)
                          "traffic": None if (awgn or offset) else measured_traffic(mode, rate, cS, cn),
                          "workload": workload_name(mode, rate, cS, cn, ", amplitude %.2f%s%s" % (
                              amp, ", AWGN sigma %.2f" % awgn if awgn else "",
                              ", constant offset -%.2f (the reference's --Xrxnoise)" % offset if offset else "")),
                          "steps": a.config_steps, "warmup": 3})
                configs.append(r)
                if cx is not cwl.x:
                    del cx
            del cwl, ceng, cfr, cst
            torch.cuda.empty_cache()

    if rank == 0:
        line = {
            "metric": METRIC,
            "value": value, "unit": "Msamples/s", "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(a.mode, a.rate, S, n,
                                                 (" (shrunk to %d streams to fit memory)" % S if shrunk else "")
                                                 + (", AWGN sigma %.2f" % a.awgn if a.awgn else "")
                                                 + (", offset -%.2f" % a.offset if a.offset else "")),
                       "streams_per_gpu": S, "nsamples": n, "frame_nsamples": frame,
                       "l2": "inputs (%.1f GB per GPU) far exceed the 126 MB L2; no flush needed" % (S * stride * 4 / 1e9),
                       "parallelism": "streams sharded over %d GPU(s); NCCL broadcast of the plan only" % world},
            "roofline": roofline, "cpu_baseline": cpu, "cpu_best_case": cpu_best, "e2e": e2e,
            "gpu_launches": int(launches),
            "clocks": clocks, "lib": mm.version(), "configs": configs,
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)


if __name__ == "__main__":
    main()
