"""Parity tests proper (B200): the CUDA path, called through the C ABI, against
the oracle on the same inputs -- the reference's own test vectors (golden
fixtures minted from the unmodified reference CLI), seeded noisy inputs, and
size-independent properties at larger batch sizes.

Bars: bits / frame_start / decoded bytes bit-exact; confidence and amplitude
within 1e-4 relative (+ the conditioning term of golden_util.close for
confidences >> 1, where two correct FFTs already disagree); inf is a class."""
import ctypes as C
import os

import numpy as np
import pytest

import golden_util as gu
import minimodem_b200 as mm
import orc
import refcases

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")


def dev():
    import conftest
    if conftest.EMU_DEVICE is not None:		# FSK_B200_EMU=1: the kernels' source on the host emulator
        return conftest.EMU_DEVICE
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda:0")


def engine_for(case_or_mode, rx=True):
    if isinstance(case_or_mode, dict):
        mode, kw = case_or_mode["rx_mode"], case_or_mode["rx_mkw"]
    else:
        mode, kw = case_or_mode
    names = dict(mark="f_mark", space="f_space", bandwidth="band_width", startbits="nstartbits",
                 stopbits="nstopbits", confidence="confidence_threshold", limit="confidence_search_limit")
    ov = {names.get(k, k): v for k, v in kw.items() if k not in ("sample_rate", "baudot")}
    if kw.get("baudot"):            # the -5 option
        ov["n_data_bits"] = 5
    cfg = mm.rx_config_for_mode(mode, kw.get("sample_rate", 48000), **ov)
    return mm.RxEngine(mm.rx_params(cfg)), cfg


def pad4(n):
    return (n + 3) & ~3


def rx_on_gpu(eng, streams, lanes=0):
    """streams: list of 1-D float32 arrays -> list of frame-record arrays."""
    n = max(len(a) for a in streams)
    stride = pad4(n)
    buf = np.zeros((len(streams), stride), np.float32)
    lens = np.zeros(len(streams), np.int32)
    for i, a in enumerate(streams):
        buf[i, :len(a)] = a
        lens[i] = len(a)
    if lanes:
        eng.tune(lanes_per_stream=lanes)
    d = torch.from_numpy(buf).to(dev())
    frames, states = eng.rx_batch(d, nsamples=n, nsamples_each=torch.from_numpy(lens).to(dev()))
    torch.cuda.synchronize()
    fr = mm.frames_to_numpy(frames)
    st = mm.states_to_numpy(states)
    assert (st["done"] == 1).all()
    return [fr[i, :st["nframes"][i]] for i in range(len(streams))], st


def as_oracle_frames(recs):
    out = []
    for r in recs:
        fs = int(r["frame_start"])
        if fs == mm.FRAME_REPORT:
            continue
        bits = int(r["bits_lo"]) | (int(r["bits_hi"]) << 32)
        out.append((bits, np.float32(r["confidence"]), np.float32(r["amplitude"]), fs & 0x7FFFFFFF,
                    1 if fs & mm.FRAME_ACQUIRED else 0, 0))
    return out


def reports_of(recs, st_row):
    """Carrier-session statistics exactly as the device accumulated them: the REPORT
    records (carrier drops, src/minimodem.c:1298-1307) plus the session still open at
    the end of the stream (:1469-1474), which lives in the stream state."""
    reps, count, nfr = [], 0, 0
    for r in recs:
        fs = int(r["frame_start"])
        if fs == mm.FRAME_REPORT:
            reps.append((count, int(r["bits_lo"]) | (int(r["bits_hi"]) << 32), np.float32(r["confidence"]),
                         np.float32(r["amplitude"]), nfr))
            count = 0
        else:
            count = 1 if fs & mm.FRAME_ACQUIRED else count + 1
            nfr += 1
    if st_row["carrier"]:
        assert int(st_row["nframes_decoded"]) == count
        reps.append((count, int(st_row["carrier_nsamples"]), np.float32(st_row["confidence_total"]),
                     np.float32(st_row["amplitude_total"]), nfr))
    return reps


def compare_reports(got, want, what=""):
    assert len(got) == len(want), (what, got, want)
    for a, b in zip(got, want):
        assert a[0] == b[0] and a[1] == b[1] and a[4] == b[4], (what, a, b)
        assert gu.close(a[2], b[2], cond=gu.CONF_COND) and gu.close(a[3], b[3]), (what, a, b)


def compare_frames(got, want, what=""):
    assert len(got) == len(want), (what, len(got), len(want))
    for i, (a, b) in enumerate(zip(got, want)):
        assert a[0] == b[0], (what, i, hex(a[0]), hex(b[0]))
        assert a[3] == b[3] and a[4] == b[4], (what, i, a, b)
        assert gu.close(a[1], b[1], cond=gu.CONF_COND), (what, i, a[1], b[1])
        assert gu.close(a[2], b[2]), (what, i, a[2], b[2])


# --------------------------------------------------------------------------
# the reference's own test vectors through the batched rx kernel
# --------------------------------------------------------------------------
RX_CASES = [c for c in refcases.EVERY]


@pytest.mark.parametrize("case", RX_CASES, ids=[c["name"] for c in RX_CASES])
def test_rx_batch_on_reference_vectors(case):
    g = gu.load(case["name"])
    _, rx = gu.modes(case)
    a = gu.audio(case, g)
    if case["rxnoise"]:
        a = (a + np.float32(-0.5) * np.float32(np.float32(case["rxnoise"]) * 2)).astype(np.float32)
    eng, cfg = engine_for(case)
    want = orc.rx_run(rx, a, literal=False, rx_one=False)
    (recs,), st = rx_on_gpu(eng, [a])
    got = as_oracle_frames(recs)
    compare_frames(got, want["frames"], case["name"])
    # byte-identical decode, the reference's own pass criterion (tests/self-test: cmp)
    frames = got
    if case["rx_one"]:          # --rx-one: stop at the first carrier drop (:1310)
        nacq = [i for i, f in enumerate(frames) if f[4]]
        if len(nacq) > 1:
            frames = frames[:nacq[1]]
    assert orc.ref_decode(rx, frames, decoder=refcases.decoder_of(case, rx)) == bytes(g["stdout"])
    # stat line (the -P tests grep it for "confidence=inf ... (rate perfect)")
    reps = reports_of(recs, st[0])
    compare_reports(reps, want["reports"], case["name"])
    lines = [orc.report_line(rx, r) for r in reps]
    wantl = gu.stat_lines(g)
    if case["rx_one"]:
        lines = lines[:1]
    assert len(lines) >= len(wantl) >= 1
    fa, fb = lines[0].split(), wantl[0].split()
    assert fa[:3] == fb[:3] and fa[4:] == fb[4:], (lines[0], wantl[0])
    assert gu.close(float(fa[3].split("=")[1]), float(fb[3].split("=")[1]), 2e-3, cond=gu.CONF_COND)
    if case["perfect"]:
        assert "confidence=inf" in lines[0] and "(rate perfect)" in lines[0]


@pytest.mark.parametrize("lanes", [4, 8, 16, 32])
@pytest.mark.parametrize("name", ["01-self-test-1200", "80-SAME", "small-rtty", "21-rate-slop-308"])
def test_rx_batch_every_lane_split(name, lanes):
    case = refcases.BY_NAME[name]
    g = gu.load(name)
    _, rx = gu.modes(case)
    a = gu.audio(case, g)
    eng, _ = engine_for(case)
    want = orc.rx_run(rx, a, literal=False)
    (recs,), _ = rx_on_gpu(eng, [a], lanes=lanes)
    compare_frames(as_oracle_frames(recs), want["frames"], "%s G=%d" % (name, lanes))


# --------------------------------------------------------------------------
# batched fsk_find_frame vs the oracle (and the compiled reference) on noisy input
# --------------------------------------------------------------------------
@pytest.mark.parametrize("mode,kw", [("1200", {}), ("300", {}), ("rtty", dict(sample_rate=8000)),
                                     ("same", {}), ("12000", {}), ("rtty", {})])
def test_find_frame_batch_noisy(mode, kw):
    m = orc.Mode(mode, **kw)
    d = m.derived()
    eng, _ = engine_for((mode, kw))
    rng = np.random.default_rng(99)
    words = rng.integers(0, 1 << m.n_data_bits, 40, dtype=np.uint32)
    clean = orc.tx_words(m, words, 1.0, 4096, True)
    spb = float(d.nsamples_per_bit)
    plan = orc.Plan(m.sample_rate, m.mark_f, m.space_f, m.band_width)
    nstreams = 256
    tmc = int(np.float32(np.float32(spb) * np.float32(0.75) + np.float32(0.5))) + d.nsamples_overscan
    tmn = int(spb) + d.nsamples_overscan
    wlen = pad4(tmn + d.expect_nsamples + int(spb) + 8)
    buf = np.zeros((nstreams, wlen), np.float32)
    args = np.zeros((nstreams, 5), np.int64)
    limit = np.zeros(nstreams, np.float32)
    sel = np.zeros(nstreams, np.uint8)
    for s in range(nstreams):
        sigma = (0.0, 0.05, 0.3, 1.0)[s % 4]
        pos = int(rng.integers(0, clean.size - wlen))
        w = clean[pos:pos + wlen] + sigma * rng.standard_normal(wlen)
        buf[s] = w.astype(np.float32)
        carrier = (s // 4) % 2
        fine = (s // 8) % 2
        tmax = tmc if carrier else tmn
        args[s] = (wlen - (s % 3) * 16, d.nsamples_overscan if carrier else 0, tmax,
                   max(tmax // (8 if fine else 3), 1), 0)
        limit[s] = np.inf if fine else 2.3
        sel[s] = 0 if carrier else 1
    t = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a.astype(dt))).to(dev())
    frames = eng.find_frame_batch(t(buf, np.float32), t(args[:, 0], np.int32), t(args[:, 1], np.int32),
                                  t(args[:, 2], np.int32), t(args[:, 3], np.int32), t(limit, np.float32),
                                  expect_sel=t(sel, np.uint8))
    torch.cuda.synchronize()
    fr = mm.frames_to_numpy(frames)
    n_bad = n_found = 0
    for s in range(nstreams):
        nv = int(args[s, 0])
        w = buf[s].copy()
        w[nv:] = 0
        expect = d.expect_data if sel[s] == 0 else d.expect_sync
        want = plan.find_frame(w, d.expect_nsamples, int(args[s, 1]), int(args[s, 2]), int(args[s, 3]),
                               float(limit[s]), expect)
        got_bits = int(fr[s]["bits_lo"]) | (int(fr[s]["bits_hi"]) << 32)
        ok = (got_bits == want[1] and int(fr[s]["frame_start"]) == want[3]
              and gu.close(fr[s]["confidence"], want[0], cond=gu.CONF_COND)
              and gu.close(fr[s]["amplitude"], want[2]))
        n_found += want[0] > 0
        if not ok:
            n_bad += 1
            assert (s % 4) != 0, (mode, s, fr[s], want)      # clean streams must match exactly
    assert n_found > nstreams // 8
    assert n_bad <= 2, n_bad                                   # razor-edge candidate flips only


# --------------------------------------------------------------------------
# the drop-in single-stream API driving the reference's rx loop
# --------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["small-1200", "small-300", "small-rtty", "small-same",
                                  "small-1200-float-noise", "70-callerid-mdmf"])
def test_dropin_find_frame_behind_the_rx_loop(name):
    """fsk_find_frame (C ABI, host buffers) plugged into the oracle's literal
    restatement of the reference rx loop, as the unmodified minimodem.c would call it."""
    case = refcases.BY_NAME[name]
    g = gu.load(name)
    _, rx = gu.modes(case)
    a = gu.audio(case, g)
    plan = mm.FskPlan(rx.sample_rate, rx.mark_f, rx.space_f, rx.band_width)
    op = orc.Plan(rx.sample_rate, rx.mark_f, rx.space_f, rx.band_width).p
    assert (plan.fftsize, plan.nbands, plan.b_mark, plan.b_space) == (op.fftsize, op.nbands, op.b_mark, op.b_space)
    L = mm.lib()

    def cb(ctx, samples, frame_nsamples, first, tmax, step, limit, expect, bits, ampl, start):
        return L.fsk_find_frame(plan._p, samples, frame_nsamples, first, tmax, step, limit, expect,
                                bits, ampl, start)

    got = orc.rx_run(rx, a, literal=True, rxnoise=case["rxnoise"], rx_one=case["rx_one"],
                     want_calls=True, find_frame=cb)
    cu, cf, cb_ = g["call_u32"], g["call_f32"], g["call_bits"]
    assert len(got["calls"]) == len(cb_)
    for i, c in enumerate(got["calls"]):
        assert c[7] == int(cb_[i]) and c[9] == int(cu[i, 4]), (i, c)
        assert gu.close(c[6], cf[i, 1], cond=gu.CONF_COND) and gu.close(c[8], cf[i, 2]), (i, c, cf[i])
    assert orc.ref_decode(rx, got["frames"]) == bytes(g["stdout"])
    plan.destroy()


def test_dropin_detect_carrier_and_bandshift():
    plan = mm.FskPlan(48000, 1200, 2200, 200)
    n = 40
    t = np.arange(n, dtype=np.float32)
    x = (0.8 * np.sin(2 * np.pi * 2200 * t / 48000)).astype(np.float32)
    assert plan.detect_carrier(x, 0.001) == 11          # 2200 Hz / 200 Hz bands
    assert plan.detect_carrier(np.zeros(n, np.float32), 0.001) == -1
    rp = orc.RefPlan(48000, 1200, 2200, 200)
    rng = np.random.default_rng(5)
    for _ in range(8):
        y = (x * rng.uniform(0.1, 1) + 0.05 * rng.standard_normal(n)).astype(np.float32)
        assert plan.detect_carrier(y, 0.001) == rp.detect_carrier(y, n, 0.001)
    plan.set_tones_by_bandshift(11, -5)                 # src/fsk.c:584-598
    assert (plan.b_mark, plan.b_space) == (11, 6)
    assert (plan.f_mark, plan.f_space) == (2200.0, 1200.0)
    plan.destroy()


@pytest.mark.parametrize("rate,bw,n", [(48000, 200.0, 40), (8000, 10.0, 176), (48000, 50.0, 160)])
def test_detect_carrier_batch(rate, bw, n):
    """N3 batched: one launch over many streams = the drop-in fsk_detect_carrier per stream
    (same band arithmetic), = the unmodified reference's pick on streams with a clear carrier."""
    plan = mm.FskPlan(rate, 1200.0 if rate == 48000 else 1585.0, 2200.0 if rate == 48000 else 1415.0, bw)
    fftsize, nbands = plan.fftsize, plan.nbands
    rng = np.random.default_rng(11)
    nstreams, stride = 70, pad4(n + 24)
    x = np.zeros((nstreams, stride), np.float32)
    off = rng.integers(0, 20, nstreams).astype(np.int32)
    t = np.arange(n, dtype=np.float32)
    bands = rng.integers(1, nbands - 1, nstreams)
    for s in range(nstreams):
        f = bands[s] * rate / fftsize
        amp = rng.uniform(0.2, 1.0)
        y = amp * np.sin(2 * np.pi * f * t / rate + rng.uniform(0, 6.28)) + 0.02 * rng.standard_normal(n)
        if s % 9 == 0:
            y = 0.0 * y                                   # silence: no band reaches the threshold
        x[s, off[s]:off[s] + n] = y.astype(np.float32)
    d = torch.from_numpy(x).to(dev())
    got = mm.detect_carrier_batch(fftsize, d, n, 0.05, offset=torch.from_numpy(off).to(dev()))
    torch.cuda.synchronize()
    got = got.cpu().numpy()
    rp = orc.RefPlan(rate, plan.f_mark, plan.f_space, bw)
    for s in range(nstreams):
        w = np.ascontiguousarray(x[s, off[s]:off[s] + n])
        assert got[s] == plan.detect_carrier(w, 0.05), s
        if s % 9 == 0:
            assert got[s] == -1
        else:
            # the window is n samples zero-padded to fftsize: the main lobe is fftsize/n bands wide
            assert abs(int(got[s]) - int(bands[s])) <= fftsize // n + 1, (s, got[s], bands[s])
        # two float DFTs may order two bands differently only when those are equal to rounding
        k = np.arange(1, nbands)[:, None] * np.arange(n)[None, :]
        m = np.abs((w[None, :].astype(np.float64) * np.exp(-2j * np.pi * k / fftsize)).sum(1))
        top = np.sort(m)[-2:]
        if top[1] == 0 or (top[1] - top[0]) / top[1] > 1e-4:
            assert got[s] == rp.detect_carrier(w, n, 0.05), s
    # no offsets, threshold above everything
    none = mm.detect_carrier_batch(fftsize, d, n, 10.0)
    torch.cuda.synchronize()
    assert (none.cpu().numpy() == -1).all()
    plan.destroy()


# --------------------------------------------------------------------------
# transmitter model on the device: bit-exact with the oracle's restatement
# --------------------------------------------------------------------------
@pytest.mark.parametrize("mode,kw", [("1200", {}), ("300", {}), ("rtty", dict(sample_rate=8000)), ("same", {})])
def test_tx_batch_bit_exact(mode, kw):
    m = orc.Mode(mode, **kw)
    eng, cfg = engine_for((mode, kw))
    rng = np.random.default_rng(3)
    nstreams, nwords = 64, 12
    words = rng.integers(0, 1 << m.n_data_bits, (nstreams, nwords), dtype=np.uint32)
    lead = rng.integers(0, 200, nstreams, dtype=np.uint32)
    tcfg = mm.tx_config_from(cfg)
    ref0 = orc.tx_words(m, words[0], 1.0, 4096, True)
    nout = ref0.size + 260
    out = mm.tx_batch(tcfg, torch.from_numpy(words.astype(np.int32)).to(dev()), nout,
                      lead_in=torch.from_numpy(lead.astype(np.int32)).to(dev()))
    torch.cuda.synchronize()
    o = out.cpu().numpy()
    for s in range(nstreams):
        want = np.zeros(nout, np.float32)
        w = orc.tx_words(m, words[s], 1.0, 4096, True)
        want[lead[s]:lead[s] + w.size] = w
        assert np.array_equal(o[s, :nout], want), s


# --------------------------------------------------------------------------
# size-independent properties on a larger batch
# --------------------------------------------------------------------------
@pytest.mark.parametrize("mode,kw,nstreams,nwords", [("1200", {}, 4096, 60), ("rtty", dict(sample_rate=8000), 2048, 20),
                                                     ("300", {}, 1024, 20), ("same", {}, 2048, 30)])
def test_roundtrip_property_large_batch(mode, kw, nstreams, nwords):
    """tx -> rx: every stream decodes exactly the words that were sent, and the same
    answer comes back for every lane split (results do not depend on the launch shape)."""
    m = orc.Mode(mode, **kw)
    d = m.derived()
    eng, cfg = engine_for((mode, kw))
    p = eng.params
    gen = torch.Generator(device="cpu").manual_seed(11)
    words = torch.randint(0, 1 << m.n_data_bits, (nstreams, nwords), generator=gen, dtype=torch.int32)
    if m.do_rx_sync:
        # no start/stop bits: the reference itself slips a bit on bytes without transitions
        # (0xFF, checked with the oracle), so use the printable payload real SAME headers carry
        words = torch.randint(32, 127, (nstreams, nwords), generator=gen, dtype=torch.int32)
    lead = torch.randint(0, int(d.nsamples_per_bit), (nstreams,), generator=gen, dtype=torch.int32)
    if m.do_rx_sync:
        # without start/stop bits the reference can lock one bit off when silence precedes the
        # periodic sync preamble (checked with the oracle); its own SAME test has no lead-in
        lead.zero_()
    tcfg = mm.tx_config_from(cfg)
    n1 = int(orc.lib().orc_tx_nsamples(C.byref(m.tx_config(1.0, 4096, True)), nwords))
    nout = n1 + int(d.nsamples_per_bit) + 8
    x = mm.tx_batch(tcfg, words.to(dev()), nout, lead_in=lead.to(dev()))
    results = []
    for lanes in (0, 32):
        eng.tune(lanes_per_stream=lanes)
        frames, states = eng.rx_batch(x, nsamples=nout)
        torch.cuda.synchronize()
        results.append((frames.clone(), states.clone()))
    # the lane split changes only the order of the fp32 correlation sums: decisions and
    # integers must agree exactly, float fields to tolerance
    fr = mm.frames_to_numpy(results[0][0])
    st = mm.states_to_numpy(results[0][1])
    fr1 = mm.frames_to_numpy(results[1][0])
    st1 = mm.states_to_numpy(results[1][1])
    assert (st["done"] == 1).all()
    for k in ("pos", "nframes", "carrier", "noconfidence", "done", "carrier_nsamples", "nframes_decoded"):
        assert np.array_equal(st[k], st1[k]), k
    assert np.allclose(st["confidence_total"], st1["confidence_total"], rtol=1e-4)
    w = words.numpy()
    shift = (1 if m.nstopbits != 0 else 0) + m.nstartbits
    mask = (1 << m.n_data_bits) - 1
    for s in range(nstreams):
        k = int(st["nframes"][s])
        for f in ("bits_lo", "bits_hi", "frame_start"):
            assert np.array_equal(fr[s, :k][f], fr1[s, :k][f]), (s, f)
        assert np.allclose(fr[s, :k]["confidence"], fr1[s, :k]["confidence"], rtol=1e-4)
        data = ((fr[s, :k]["bits_lo"].astype(np.uint64) | (fr[s, :k]["bits_hi"].astype(np.uint64) << np.uint64(32)))
                >> np.uint64(shift)) & np.uint64(mask)
        if m.do_rx_sync:
            data = data[data != (m.sync_byte & mask)]
        # the leader/trailer may add idle frames around the payload; the payload must be inside
        got = data.astype(np.int64).tolist()
        want = (w[s] & mask).tolist()
        assert any(got[i:i + len(want)] == want for i in range(len(got) - len(want) + 1)), (s, got, want)
    # cross-check a sample of streams frame by frame against the oracle
    xs = x[:16].cpu().numpy()
    for s in range(16):
        want = orc.rx_run(m, xs[s, :nout], literal=False)
        compare_frames(as_oracle_frames(fr[s, :st["nframes"][s]]), want["frames"], "stream %d" % s)


# --------------------------------------------------------------------------
# BASELINE config 4: Bell103 300 baud with a noise sweep, confidence match vs the CPU
# --------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["offset", "awgn"])
def test_bell103_noise_sweep_confidence_match(kind):
    """The reference's --Xrxnoise quirk (a constant -f offset, src/simpleaudio-sndfile.c:64-70)
    and true additive noise at the same levels: every frame of every stream must carry the
    oracle's bits / frame_start, and its confidence within tolerance."""
    m = orc.Mode("300")
    eng, cfg = engine_for(("300", {}))
    rng = np.random.default_rng(40)
    levels = [0.0, 0.05, 0.10, 0.50]
    streams = []
    for s in range(64):
        words = rng.integers(32, 127, 24, dtype=np.uint32)
        x = orc.tx_words(m, words, 0.5, 4096, True)          # --volume 0.5 as tests/40-noise.test
        lead = int(rng.integers(0, 160))
        x = np.concatenate([np.zeros(lead, np.float32), x])
        f = levels[s % 4]
        if kind == "offset":
            x = (x + np.float32(-0.5) * np.float32(np.float32(f) * 2)).astype(np.float32)
        else:
            x = (x + f * 0.5 * rng.standard_normal(x.size)).astype(np.float32)
        streams.append(x)
    recs, st = rx_on_gpu(eng, streams)
    n_frames = n_flip = 0
    for s, x in enumerate(streams):
        want = orc.rx_run(m, x, literal=False)
        got = as_oracle_frames(recs[s])
        n_frames += len(want["frames"])
        try:
            compare_frames(got, want["frames"], "%s stream %d" % (kind, s))
            compare_reports(reports_of(recs[s], st[s]), want["reports"], "%s stream %d" % (kind, s))
        except AssertionError:
            # a razor-edge early-out flip (|confidence - limit| ~ 1e-7) is legitimate on noisy
            # input, but it must stay an exception and the decoded data must still agree
            n_flip += 1
            assert levels[s % 4] > 0 and kind == "awgn", (kind, s)
            assert [orc.databits(m, f[0]) for f in got] == [orc.databits(m, f[0]) for f in want["frames"]]
    assert n_frames > 64 * 20
    assert n_flip <= 1


# --------------------------------------------------------------------------
# edge cases: empty / short / ragged streams, silence, noise only, output overflow + resume
# --------------------------------------------------------------------------
def test_rx_batch_edge_cases_ragged_batch():
    m = orc.Mode("1200")
    eng, cfg = engine_for(("1200", {}))
    rng = np.random.default_rng(8)
    base = orc.tx_words(m, rng.integers(32, 127, 30, dtype=np.uint32), 1.0, 4096, True)
    d = m.derived()
    streams = [
        np.zeros(0, np.float32),                              # empty
        base[:d.expect_nsamples - 1].copy(),                  # one sample short of a search window (:1229)
        base[:d.expect_nsamples].copy(),                      # exactly one window
        np.zeros(5000, np.float32),                           # silence: never any carrier
        (0.3 * rng.standard_normal(20000)).astype(np.float32),   # noise only
        base.copy(),                                          # a normal stream
        base[:base.size // 2 + 7].copy(),                     # cut in the middle of a frame
        np.concatenate([base, np.zeros(3000, np.float32), base]).astype(np.float32),   # carrier drop + re-acquire
        (base * np.float32(1e-6)).astype(np.float32),         # tiny amplitude: confidence is scale free
    ]
    for lanes in (0, 16):
        recs, st = rx_on_gpu(eng, streams, lanes=lanes)
        for s, x in enumerate(streams):
            want = orc.rx_run(m, x, literal=False)
            compare_frames(as_oracle_frames(recs[s]), want["frames"], "edge stream %d (G=%d)" % (s, lanes))
            compare_reports(reports_of(recs[s], st[s]), want["reports"], "edge stream %d (G=%d)" % (s, lanes))
    assert len(recs[0]) == 0 and len(recs[1]) == 0 and len(recs[3]) == 0
    assert sum(1 for r in recs[7] if int(r["frame_start"]) == mm.FRAME_REPORT) == 1


def test_rx_batch_output_overflow_and_resume():
    """A stream that fills its record buffer stops with done=0 and can be continued from its
    saved state; the concatenated records equal those of an unbounded run."""
    m = orc.Mode("1200")
    eng, cfg = engine_for(("1200", {}))
    rng = np.random.default_rng(9)
    xs = [orc.tx_words(m, rng.integers(32, 127, 40, dtype=np.uint32), 1.0, 4096, True) for _ in range(5)]
    n = max(len(a) for a in xs)
    buf = np.zeros((len(xs), pad4(n)), np.float32)
    for i, a in enumerate(xs):
        buf[i, :len(a)] = a
    d = torch.from_numpy(buf).to(dev())
    lens = torch.from_numpy(np.array([len(a) for a in xs], np.int32)).to(dev())
    full, st_full = eng.rx_batch(d, nsamples=n, nsamples_each=lens)
    small, st = eng.rx_batch(d, nsamples=n, nsamples_each=lens, max_frames=10)
    torch.cuda.synchronize()
    s1 = mm.states_to_numpy(st)
    assert (s1["done"] == 0).all() and (s1["nframes"] == 10).all()
    big = torch.zeros_like(full)
    _, st2 = eng.rx_batch(d, nsamples=n, nsamples_each=lens, max_frames=full.shape[1], frames=big, states=st)
    torch.cuda.synchronize()
    f_full, f_small, f_big = (mm.frames_to_numpy(t) for t in (full, small, big))
    sf, s2 = mm.states_to_numpy(st_full), mm.states_to_numpy(st2)
    assert (s2["done"] == 1).all() and np.array_equal(s2["nframes"], sf["nframes"])
    for i in range(len(xs)):
        k = int(sf["nframes"][i])
        joined = np.concatenate([f_small[i, :10], f_big[i, 10:k]])
        assert np.array_equal(joined, f_full[i, :k]), i
    for key in ("pos", "carrier", "carrier_nsamples", "nframes_decoded", "confidence_total", "amplitude_total"):
        assert np.array_equal(s2[key], sf[key]), key


def test_find_frame_batch_degenerate_arguments():
    eng, cfg = engine_for(("1200", {}))
    p = eng.params
    nstreams = 7                                              # not a multiple of anything
    w = pad4(p.try_max_nocarrier + p.span_nsamples + 8)
    x = torch.zeros((nstreams, w), dtype=torch.float32, device=dev())
    i32 = lambda v: torch.full((nstreams,), v, dtype=torch.int32, device=dev())
    tmax = i32(p.try_max_nocarrier)
    tmax[0] = 0                                               # empty search range: loop never runs (:481)
    nv = i32(w)
    nv[1] = 0                                                 # no valid samples at all
    fr = eng.find_frame_batch(x, nv, i32(0), tmax, i32(0), torch.full((nstreams,), 2.3, device=dev()))
    torch.cuda.synchronize()
    f = mm.frames_to_numpy(fr)
    # silence: every bit ties (mag_mark == mag_space == 0 -> space), the start bit pattern mismatches
    assert (f["confidence"] == 0).all() and (f["bits_lo"] == 0).all() and (f["frame_start"] == 0).all()


# --------------------------------------------------------------------------
# "next" rows: N2 16-bit PCM ingest, N1 on-device ASCII databits decode
# --------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["01-self-test-1200", "02-self-test-300", "80-SAME", "81-ascii7", "60-multibyte"])
def test_s16_ingest_and_device_ascii_decode(name):
    """The reference transmitter's default format is S16; its rx reads short/32768
    (src/simpleaudio-sndfile.c:43-57).  The int16 host path must give exactly the records of the
    float path, and the device decoder exactly the bytes the reference printed."""
    case = refcases.BY_NAME[name]
    g = gu.load(name)
    _, rx = gu.modes(case)
    a = gu.audio(case, g)
    s16 = np.round(a * 32768.0).astype(np.int16)
    assert np.array_equal(s16.astype(np.float32) * np.float32(1 / 32768.0), a)     # vectors really are S16
    eng, cfg = engine_for(case)
    n = a.size
    stride = pad4(n)
    nstreams = 3
    hs = np.zeros((nstreams, stride), np.int16)
    hf = np.zeros((nstreams, stride), np.float32)
    hs[:, :n] = s16
    hf[:, :n] = a
    fr_f, st_f = eng.rx_batch_host(hf, nsamples=n)
    fr_s, st_s = eng.rx_batch_host_s16(hs, nsamples=n)
    assert np.array_equal(st_f, st_s)
    k = int(st_f["nframes"][0])
    assert k > 0 and np.array_equal(fr_f[:, :k], fr_s[:, :k])
    # device conversion kernel on its own
    d = mm.s16_to_f32(torch.from_numpy(hs).to(dev()))
    torch.cuda.synchronize()
    assert np.array_equal(d.cpu().numpy(), hf)
    # device decode of the device-resident records
    frames, states = eng.rx_batch(d, nsamples=n)
    out, cnt = eng.decode_ascii_batch(frames, states)
    torch.cuda.synchronize()
    o, c = out.cpu().numpy(), cnt.cpu().numpy()
    want = bytes(g["stdout"])
    for s in range(nstreams):
        assert bytes(o[s, :c[s]]) == want, s


# --------------------------------------------------------------------------
# N1: every databits decoder on the device (k_decode<KIND>) against the host build of the
# same source (oracle/decode_oracle.c), which test_decoders.py pins to the reference decoders
# --------------------------------------------------------------------------
DEC_MODES = {"ascii8": ("1200", {}), "binary": ("1200", {}), "baudot": ("rtty", dict(sample_rate=8000)),
             "callerid": ("callerid", {}), "uic-ground": ("uic-ground", {}), "uic-train": ("uic-train", {})}


def _synthetic_records(kind, rx, rng, nstreams, max_frames):
    """Frame records a demodulator could have written: data words under the mode's framing, a
    carrier acquire here and there, session reports in between, ragged record counts."""
    nb = rx.n_data_bits
    shift = (1 if rx.nstopbits != 0.0 else 0) + int(rx.nstartbits)
    rec = np.zeros((nstreams, max_frames, 5), np.uint32)
    nfr = rng.integers(0, max_frames + 1, nstreams).astype(np.uint32)
    nfr[:4] = [0, 1, max_frames, max_frames]
    for s in range(nstreams):
        n = int(nfr[s])
        if kind == "callerid":
            # byte traffic with frequent message starts and short lengths, so that messages complete
            w = rng.integers(0, 256, n, dtype=np.uint64)
            i = 0
            while i + 2 < n:
                ln = int(rng.integers(0, 24))
                w[i] = int(rng.choice([0x80, 0x04]))
                w[i + 1] = ln
                if w[i] == 0x80:
                    j = i + 2
                    while j + 2 <= min(n, i + 2 + ln):
                        w[j] = int(rng.choice([1, 2, 4, 7, 8, 3, 9]))
                        fl = int(min(rng.integers(0, 11), i + 2 + ln - j - 2))
                        w[j + 1] = fl
                        j += 2 + fl
                i += ln + 3 + int(rng.integers(0, 3))
        elif kind == "baudot":
            w = rng.integers(0, 32, n, dtype=np.uint64)
        else:
            w = rng.integers(0, 1 << min(nb, 62), n, dtype=np.uint64)
        junk = rng.integers(0, 1 << 62, n, dtype=np.uint64)
        mask = np.uint64(((1 << nb) - 1) << shift)
        bits = ((w << np.uint64(shift)) & mask) | (junk & ~mask)       # framing bits are arbitrary
        if rx.frame_n_bits + 1 < 64:
            bits &= np.uint64((1 << (rx.frame_n_bits + 1)) - 1)
        rec[s, :n, 0] = (bits & np.uint64(0xFFFFFFFF)).astype(np.uint32)
        rec[s, :n, 1] = (bits >> np.uint64(32)).astype(np.uint32)
        rec[s, :n, 4] = rng.integers(0, 100, n).astype(np.uint32)
        acq = rng.random(n) < 0.03
        if n:
            acq[0] = True
        rec[s, :n, 4] |= np.where(acq, orc.FRAME_ACQUIRED, 0).astype(np.uint32)
        rep = rng.random(n) < 0.02
        rec[s, :n, 4] = np.where(rep, orc.FRAME_REPORT, rec[s, :n, 4])
    return rec, nfr


@pytest.mark.parametrize("kind", list(DEC_MODES))
def test_decode_batch_every_decoder(kind):
    mode, kw = DEC_MODES[kind]
    rx = orc.Mode(mode, **kw)
    eng, _ = engine_for((mode, kw))
    k = orc.DECODE_KINDS[kind]
    assert mm.decoder_for_mode(mode, rx.n_data_bits, binary_output=(kind == "binary")) == k
    rng = np.random.default_rng(100 + k)
    nstreams, max_frames = 700, 96
    rec, nfr = _synthetic_records(kind, rx, rng, nstreams, max_frames)
    st = np.zeros(nstreams, mm.STATE_DTYPE)
    st["nframes"] = nfr
    d_rec = torch.from_numpy(rec.view(np.int32)).to(dev())
    d_st = torch.from_numpy(st.view(np.int32).reshape(nstreams, -1)).to(dev())
    out, cnt = eng.decode_batch(k, d_rec, d_st)
    torch.cuda.synchronize()
    o, c = out.cpu().numpy(), cnt.cpu().numpy()
    total = 0
    for s in range(nstreams):
        want = orc.decode_records(rx, kind, rec[s, :nfr[s]])
        assert bytes(o[s, :c[s]]) == want, (kind, s)
        total += len(want)
    assert total > 1000
    # independent of this repository's decoder source: the UNMODIFIED reference decoders (oracle/_ref/libfsk_ref.so,
    # src/databits_*.c, src/uic_codes.c) on the same records, for the decoders that keep no state between calls
    if kind in ("ascii8", "binary", "uic-ground", "uic-train"):
        for s in range(0, nstreams, 5):
            frames = []
            for r in rec[s, :nfr[s]]:
                if int(r[4]) == orc.FRAME_REPORT:
                    continue
                frames.append((int(r[0]) | (int(r[1]) << 32), 0.0, 0.0, int(r[4]) & 0x7FFFFFFF,
                               1 if int(r[4]) & orc.FRAME_ACQUIRED else 0, 0))
            assert bytes(o[s, :c[s]]) == orc.ref_decode(rx, frames, decoder=kind), (kind, s, "vs the reference decoder")

    # the same streams in two batches with the decoder state carried on the device
    half = max_frames // 2
    dst = torch.zeros((nstreams, mm.DECODER_STATE_BYTES), dtype=torch.uint8, device=dev())
    st1 = st.copy()
    st1["nframes"] = np.minimum(nfr, half)
    st2 = st.copy()
    st2["nframes"] = nfr - st1["nframes"]
    rec2 = np.zeros_like(rec)
    rec2[:, :max_frames - half] = rec[:, half:]
    o1, c1 = eng.decode_batch(k, d_rec, torch.from_numpy(st1.view(np.int32).reshape(nstreams, -1)).to(dev()), dstates=dst)
    o2, c2 = eng.decode_batch(k, torch.from_numpy(rec2.view(np.int32)).to(dev()),
                              torch.from_numpy(st2.view(np.int32).reshape(nstreams, -1)).to(dev()), dstates=dst)
    torch.cuda.synchronize()
    o1, c1, o2, c2 = o1.cpu().numpy(), c1.cpu().numpy(), o2.cpu().numpy(), c2.cpu().numpy()
    for s in range(nstreams):
        assert bytes(o1[s, :c1[s]]) + bytes(o2[s, :c2[s]]) == bytes(o[s, :c[s]]), (kind, s)

    # a short output row: the count is clamped, the stored prefix is intact
    o3, c3 = eng.decode_batch(k, d_rec, d_st, out_stride=7)
    torch.cuda.synchronize()
    o3, c3 = o3.cpu().numpy(), c3.cpu().numpy()
    for s in range(0, nstreams, 37):
        assert c3[s] == min(c[s], 7) and bytes(o3[s, :c3[s]]) == bytes(o[s, :c3[s]])


@pytest.mark.parametrize("name", ["03-self-test-rtty", "81-tdd", "70-callerid-mdmf", "71-callerid-sdmf", "small-rtty"])
def test_rx_then_device_decode_prints_what_the_reference_printed(name):
    """Samples in, text out, all on the device: rx_batch + decode_batch with the decoder the
    reference's main() picks for the mode = the stdout of the unmodified reference CLI."""
    case = refcases.BY_NAME[name]
    g = gu.load(name)
    _, rx = gu.modes(case)
    a = gu.audio(case, g)
    eng, cfg = engine_for(case)
    n = a.size
    buf = np.zeros((2, pad4(n)), np.float32)
    buf[:, :n] = a
    frames, states = eng.rx_batch(torch.from_numpy(buf).to(dev()), nsamples=n)
    kind = mm.decoder_for_mode(case["rx_mode"], rx.n_data_bits)
    out, cnt = eng.decode_batch(kind, frames, states)
    torch.cuda.synchronize()
    o, c = out.cpu().numpy(), cnt.cpu().numpy()
    for s in range(2):
        assert bytes(o[s, :c[s]]) == bytes(g["stdout"]), s


def test_uic_frames_end_to_end():
    """UIC-751-3 (src/minimodem.c:859-875): 47-bit frames behind the fixed pattern 11110010, the
    longest expect string of the reference.  It has no transmitter there, so the stream is made bit
    by bit with the oracle's tone generator; samples in, text out on the device."""
    rx = orc.Mode("uic-ground")
    bitm = orc.Mode("600", mark=rx.mark_f, space=rx.space_f, n_data_bits=1, startbits=0, stopbits=0.0)

    def frame_bits(train, code):
        word = train | (int("{:08b}".format(code)[::-1], 2) << 24)
        return [int(c) for c in "11110010"] + [(word >> i) & 1 for i in range(39)]

    msgs = [(0x123456, 0x09), (0x654321, 0x55), (0xABCDEF, 0x02), (0x000001, 0x7E), (0x13579B, 0x0C)]
    rng = np.random.default_rng(21)
    streams = []
    for s in range(4):
        bits = [1] * int(rng.integers(12, 40))
        for t, c in msgs[s:] + msgs[:s]:
            bits += frame_bits(t, c)                          # frames follow each other directly
        bits += [1] * 30
        a = orc.tx_words(bitm, np.array(bits, np.uint32), float(rng.uniform(0.4, 1.0)), 4096, True)
        streams.append((a + np.float32(0.005) * rng.standard_normal(a.size).astype(np.float32)).astype(np.float32))
    for mode, kind in (("uic-ground", mm.DECODE_UIC_GROUND), ("uic-train", mm.DECODE_UIC_TRAIN)):
        eng, _ = engine_for((mode, {}))
        n = max(len(a) for a in streams)
        buf = np.zeros((len(streams), pad4(n)), np.float32)
        lens = np.zeros(len(streams), np.int32)
        for i, a in enumerate(streams):
            buf[i, :len(a)] = a
            lens[i] = len(a)
        frames, states = eng.rx_batch(torch.from_numpy(buf).to(dev()), nsamples=n,
                                      nsamples_each=torch.from_numpy(lens).to(dev()))
        out, cnt = eng.decode_batch(kind, frames, states)
        torch.cuda.synchronize()
        fr, st = mm.frames_to_numpy(frames), mm.states_to_numpy(states)
        o, c = out.cpu().numpy(), cnt.cpu().numpy()
        for s, a in enumerate(streams):
            want = orc.rx_run(rx, a, literal=False)
            compare_frames(as_oracle_frames(fr[s, :st["nframes"][s]]), want["frames"], "%s stream %d" % (mode, s))
            text = bytes(o[s, :c[s]])
            assert text == orc.decode_records(rx, "uic-ground" if kind == mm.DECODE_UIC_GROUND else "uic-train",
                                              orc.frame_records(want["frames"]))
            assert text.count(b"Train ID: ") == len(msgs), text
        if kind == mm.DECODE_UIC_GROUND:
            assert b"Train ID: 654321 - Message: 09 (Emergency stop)\n" in bytes(o[0, :c[0]])


@pytest.mark.parametrize("fmt", ["f32", "s16"])
def test_host_buffer_path_in_many_slabs(fmt, monkeypatch):
    """fsk_b200_rx_batch_host splits a batch into slabs (256 MiB on the wire by default) and keeps two in
    flight; with the slab shrunk to two float streams (four int16 ones), 7 streams take 4 (2) slabs, the
    last one partial, on alternating buffers -- records and states must equal the one-launch device
    path, stream by stream."""
    case = refcases.BY_NAME["small-1200"]
    g = gu.load(case["name"])
    a = gu.audio(case, g)
    rng = np.random.default_rng(2)
    n = a.size + 600
    stride = pad4(n)
    nstreams = 7
    hf = np.zeros((nstreams, stride), np.float32)
    for s in range(nstreams):
        lead = int(rng.integers(0, 600))
        hf[s, lead:lead + a.size] = a * np.float32(rng.integers(2, 9) / 8.0)
    hs = np.round(hf * 32768.0).astype(np.int16)
    hf = hs.astype(np.float32) * np.float32(1 / 32768.0)       # the float streams ARE the int16 ones
    monkeypatch.setenv("FSK_B200_SLAB_BYTES", str(2 * stride * 4))
    eng, _ = engine_for(case)
    monkeypatch.delenv("FSK_B200_SLAB_BYTES")
    ref_eng, _ = engine_for(case)
    frames, states = ref_eng.rx_batch(torch.from_numpy(hf).to(dev()), nsamples=n)
    torch.cuda.synchronize()
    want_fr, want_st = mm.frames_to_numpy(frames), mm.states_to_numpy(states)
    if fmt == "f32":
        fr, st = eng.rx_batch_host(hf, nsamples=n)
    else:
        fr, st = eng.rx_batch_host_s16(hs, nsamples=n)
    assert np.array_equal(st, want_st)
    for s in range(nstreams):
        k = int(want_st["nframes"][s])
        assert k > 0 and np.array_equal(fr[s, :k], want_fr[s, :k]), s


# --------------------------------------------------------------------------
# the drop-in boundary end to end: the unmodified reference CLI on this library
# --------------------------------------------------------------------------
def _write_wav(path, samples, rate, as_float):
    import struct
    if as_float:
        data, fmt, bits = samples.astype("<f4").tobytes(), 3, 32
    else:
        data, fmt, bits = np.round(samples * 32768.0).astype("<i2").tobytes(), 1, 16
    hdr = b"RIFF" + struct.pack("<I", 36 + len(data)) + b"WAVE" + b"fmt " + struct.pack(
        "<IHHIIHH", 16, fmt, 1, rate, rate * bits // 8, bits // 8, bits) + b"data" + struct.pack("<I", len(data))
    with open(path, "wb") as f:
        f.write(hdr + data)


CLI_CASES = [c for c in refcases.EVERY + refcases.CLI_ONLY if c["audio"]]


@pytest.mark.parametrize("case", CLI_CASES, ids=[c["name"] for c in CLI_CASES])
def test_reference_cli_on_this_library(case, tmp_path):
    """oracle/_ref/minimodem_dropin = the reference's own main(), rx loop, decoders and src/fsk.h,
    compiled unmodified and linked against libfsk_b200.so instead of src/fsk.c + FFTW.  On the
    audio of the committed vectors it must print what the reference printed: stdout byte for byte,
    the stat lines field for field (confidence to tolerance)."""
    import os
    import subprocess
    import conftest
    exe = os.path.join(os.path.dirname(orc.LIBREF), "minimodem_dropin")
    if not os.path.exists(exe):
        pytest.skip("oracle/_ref/minimodem_dropin not built (needs /root/reference at build time)")
    g = gu.load(case["name"])
    a = gu.audio(case, g)
    rate = int(g["audio_len"][1])
    wav = str(tmp_path / "x.wav")
    _write_wav(wav, a, rate, bool(g["audio_len"][2]))
    env = dict(os.environ)
    if conftest.EMU_DEVICE is not None:         # FSK_B200_EMU=1: the emulation build answers to the library's name
        import test_dropin_cli
        env["LD_LIBRARY_PATH"] = test_dropin_cli.emulation_as_product()
    r = subprocess.run([exe, "--rx", "--file", wav] + list(case["rx"]), env=env, stdout=subprocess.PIPE,
                       stderr=subprocess.PIPE, timeout=600)
    assert r.returncode == 0, r.stderr[-500:]
    assert r.stdout == bytes(g["stdout"])
    got = [ln for ln in r.stderr.decode().splitlines() if ln.startswith("### NOCARRIER")]
    want = gu.stat_lines(g)
    assert len(got) == len(want)
    for x, y in zip(got, want):
        fa, fb = x.split(), y.split()
        assert fa[:3] == fb[:3] and fa[4:] == fb[4:], (x, y)
        ca, cb = float(fa[3].split("=")[1]), float(fb[3].split("=")[1])
        assert gu.close(ca, cb, 2e-3, cond=gu.CONF_COND) or (np.isinf(ca) and np.isinf(cb)), (x, y)


def test_batched_entry_points_reject_bad_arguments():
    """EINVAL with a message, never a launch: rows that are not 16-byte aligned, missing output
    arrays, zero-sized record buffers, unknown decoders, detect windows longer than the transform."""
    import errno
    eng, cfg = engine_for(("1200", {}))
    L = mm.lib()
    x = torch.zeros((4, 4096), dtype=torch.float32, device=dev())
    fr = torch.zeros((4, 16, 5), dtype=torch.int32, device=dev())
    st = torch.zeros((4, mm.STATE_WORDS), dtype=torch.int32, device=dev())
    p = lambda t: C.c_void_p(t.data_ptr())
    before = mm.launch_count()
    bad = [
        L.fsk_b200_rx_batch(eng._e, p(x), 4, 4095, None, 4095, p(fr), 16, p(st), None),       # stride % 4
        L.fsk_b200_rx_batch(eng._e, C.c_void_p(x.data_ptr() + 4), 4, 4092, None, 4000, p(fr), 16, p(st), None),
        L.fsk_b200_rx_batch(eng._e, p(x), 4, 4096, None, 4096, None, 16, p(st), None),        # no record array
        L.fsk_b200_rx_batch(eng._e, p(x), 4, 4096, None, 4096, p(fr), 0, p(st), None),        # no room for records
        L.fsk_b200_rx_batch(eng._e, None, 4, 4096, None, 4096, p(fr), 16, p(st), None),
        L.fsk_b200_decode_batch(C.byref(eng.params), 17, p(fr), p(st), 4, 16, None, p(x), 64, p(st), None),
        L.fsk_b200_decode_batch(C.byref(eng.params), 0, p(fr), p(st), 4, 16, None, p(x), 0, p(st), None),
        L.fsk_b200_detect_carrier_batch(240, p(x), 4, 4096, None, 241, 0.1, p(st), None),
        L.fsk_b200_detect_carrier_batch(240, p(x), 4, 4096, None, 0, 0.1, p(st), None),
    ]
    assert all(rc == -errno.EINVAL for rc in bad), bad
    assert L.fsk_b200_last_error()
    assert mm.launch_count() == before
    assert L.fsk_b200_rx_batch(eng._e, p(x), 0, 4096, None, 4096, p(fr), 16, p(st), None) == 0   # empty batch


# --------------------------------------------------------------------------
# live streams: chunked feeding with carry-over == one pass over the whole stream
# --------------------------------------------------------------------------
@pytest.mark.parametrize("mode,kw", [("1200", {}), ("300", {}), ("rtty", dict(sample_rate=8000)), ("same", {})])
def test_streams_fed_in_chunks_give_the_records_of_one_pass(mode, kw):
    """fsk_b200_stream_push + fsk_b200_engine_set_holdback: every stream gets its samples in chunks of
    its own random sizes (down to a handful of samples), keeps what the loop has not consumed, and is
    flushed at the end with the reference's end-of-input rule.  The concatenated records must be
    those of a single pass over the complete stream -- identical, not merely close: the same kernel
    sees the same samples in the same windows."""
    rx = orc.Mode(mode, **kw)
    d = rx.derived()
    rng = np.random.default_rng(31)
    nstreams = 6
    full = []
    for s in range(nstreams):
        parts = [np.zeros(int(rng.integers(0, 3 * int(d.nsamples_per_bit))), np.float32)]
        for _ in range(int(rng.integers(1, 4))):
            w = rng.integers(0, 1 << rx.n_data_bits, int(rng.integers(3, 14)), dtype=np.uint64).astype(np.uint32)
            parts.append(orc.tx_words(rx, w, float(rng.uniform(0.3, 1.0)), 4096, True))
            parts.append(np.zeros(int(rng.integers(0, 40)) * int(d.nsamples_per_bit), np.float32))
        x = np.concatenate(parts).astype(np.float32)
        full.append((x + np.float32(0.004) * rng.standard_normal(x.size).astype(np.float32)).astype(np.float32))
    eng, _ = engine_for((mode, kw))
    # one pass
    want, st_want = rx_on_gpu(eng, full)
    # chunked
    window = eng.stream_window()
    assert window == eng.params.try_max_nocarrier - 1 + eng.params.span_nsamples
    max_chunk = 3 * window
    stride = pad4(window + 2 * max_chunk + 64)
    rows = torch.zeros((nstreams, stride), dtype=torch.float32, device=dev())
    fill = torch.zeros((nstreams,), dtype=torch.int32, device=dev())
    states = torch.zeros((nstreams, mm.STATE_WORDS), dtype=torch.int32, device=dev())
    dropped = torch.zeros((nstreams,), dtype=torch.int32, device=dev())
    eng.set_holdback(window)
    fed = [0] * nstreams
    got = [[] for _ in range(nstreams)]
    max_frames = eng.max_frames(stride)

    def collect(frames, st):
        fr, s1 = mm.frames_to_numpy(frames), mm.states_to_numpy(st)
        for i in range(nstreams):
            got[i].extend(fr[i, :s1["nframes"][i]].copy())
        return s1

    for _ in range(10000):
        if all(fed[i] >= len(full[i]) for i in range(nstreams)):
            break
        chunk = np.zeros((nstreams, max_chunk), np.float32)
        clen = np.zeros(nstreams, np.int32)
        for i in range(nstreams):
            k = int(min(rng.integers(1, max_chunk + 1) if rng.random() < 0.8 else rng.integers(1, 9),
                        len(full[i]) - fed[i]))
            chunk[i, :k] = full[i][fed[i]:fed[i] + k]
            clen[i] = k
            fed[i] += k
        mm.stream_push(rows, fill, states, torch.from_numpy(chunk).to(dev()), torch.from_numpy(clen).to(dev()),
                       dropped=dropped)
        frames, states = eng.rx_batch(rows, nsamples=stride, nsamples_each=fill, max_frames=max_frames, states=states)
        torch.cuda.synchronize()
        assert int(dropped.sum()) == 0
        collect(frames, states)
    else:
        raise AssertionError("feeding did not finish")
    # end of input: the reference's rule takes over (src/minimodem.c:1229)
    eng.set_holdback(0)
    mm.stream_push(rows, fill, states, torch.zeros((nstreams, 4), dtype=torch.float32, device=dev()), 0)
    frames, states = eng.rx_batch(rows, nsamples=stride, nsamples_each=fill, max_frames=max_frames, states=states)
    torch.cuda.synchronize()
    s_end = collect(frames, states)
    assert (s_end["done"] == 1).all()
    # The per-candidate and shared-segment kernels count the correlation phase from the window (or bit period), so
    # the arithmetic does not depend on where a stream sits in its row: identical records.  The prefix-table kernel
    # counts it from the 16-byte chunk that holds the search position, and stream_push moves that: the same sums in
    # another rounding (a few 1e-7 relative), so bits and positions must still be identical, the statistics close.
    exact = "prefix-table" not in eng.last_kernel()
    for i in range(nstreams):
        a = np.array(got[i], dtype=mm.FRAME_DTYPE) if got[i] else np.zeros(0, mm.FRAME_DTYPE)
        if exact:
            assert np.array_equal(a, want[i]), (mode, i, len(a), len(want[i]))
            continue
        assert len(a) == len(want[i]), (mode, i, len(a), len(want[i]))
        for key in ("bits_lo", "bits_hi", "frame_start"):
            assert np.array_equal(a[key], want[i][key]), (mode, i, key)
        for key in ("confidence", "amplitude"):
            assert np.allclose(a[key], want[i][key], rtol=2e-5, atol=0), (mode, i, key)
    for key in ("carrier", "carrier_nsamples", "nframes_decoded", "confidence_total", "amplitude_total",
                "noconfidence", "track_amplitude", "peak_confidence"):
        if exact or key in ("carrier", "carrier_nsamples", "nframes_decoded", "noconfidence"):
            assert np.array_equal(s_end[key], st_want[key]), key
        else:
            assert np.allclose(s_end[key], st_want[key], rtol=2e-5, atol=0), key


@pytest.mark.parametrize("name", ["small-rtty", "70-callerid-mdmf", "71-callerid-sdmf", "small-same", "small-1200",
                                  "opt-sync-byte-600"])
def test_live_receiver_prints_the_reference_output_however_the_stream_is_cut(name):
    """minimodem_b200.LiveReceiver (stream_push -> rx_batch -> decode_batch, all on the device): the
    audio of a reference vector fed in random chunks -- a different cut for every stream -- must add
    up to what the unmodified reference CLI printed for the whole file."""
    case = refcases.BY_NAME[name]
    g = gu.load(name)
    _, rx = gu.modes(case)
    a = gu.audio(case, g)
    rng = np.random.default_rng(77)
    nstreams, max_chunk = 4, 2048
    names = dict(mark="f_mark", space="f_space", bandwidth="band_width", startbits="nstartbits", stopbits="nstopbits")
    ov = {names.get(k, k): v for k, v in case["rx_mkw"].items() if k != "sample_rate"}
    lr = mm.LiveReceiver(case["rx_mode"], sample_rate=rx.sample_rate, nstreams=nstreams, max_chunk=max_chunk,
                         device=dev(), **ov)
    fed = [0] * nstreams
    text = [bytearray() for _ in range(nstreams)]

    def take(out, cnt):
        o, c = out.cpu().numpy(), cnt.cpu().numpy()
        for i in range(nstreams):
            text[i] += bytes(o[i, :c[i]])

    while any(f < a.size for f in fed):
        chunk = np.zeros((nstreams, max_chunk), np.float32)
        clen = np.zeros(nstreams, np.int32)
        for i in range(nstreams):
            k = int(min(rng.integers(1, max_chunk + 1) if i else max_chunk, a.size - fed[i]))
            if i == 1:
                k = min(k, 333)                                # one stream trickles in
            chunk[i, :k] = a[fed[i]:fed[i] + k]
            clen[i] = k
            fed[i] += k
        take(*lr.feed(torch.from_numpy(chunk).to(dev()), torch.from_numpy(clen).to(dev())))
    take(*lr.finish())
    torch.cuda.synchronize()
    assert int(lr.dropped.sum()) == 0
    for i in range(nstreams):
        assert bytes(text[i]) == bytes(g["stdout"]), i


# --------------------------------------------------------------------------
# per-bit parity gate (BASELINE.md 3, SURVEY.md 7 hard part 3): what fsk_bit_analyze saw in every
# bit window of the winning candidate -- signal and noise magnitudes of src/fsk.c:158-169 --
# against the oracle's: rel 1e-4 on the signal, abs 1e-4 * (mean signal) on the noise, and the
# noise <= FLT_EPSILON class of :278-280 (what makes `confidence=inf`) exactly
# --------------------------------------------------------------------------
PERBIT_MODES = [("1200", {}), ("rtty", dict(sample_rate=8000)), ("300", {}), ("same", {}),
                ("1200", dict(mark=1200, space=2400))]          # the last: orthogonal tones, the -P vectors' geometry


@pytest.mark.parametrize("mode,kw", PERBIT_MODES, ids=["cfg2-1200", "cfg3-rtty8k", "cfg4-bell103", "cfg5-same", "purefreqs"])
def test_per_bit_magnitudes_vs_oracle(mode, kw):
    m = orc.Mode(mode, **kw)
    d = m.derived()
    eng, _ = engine_for((mode, kw))
    rng = np.random.default_rng(7)
    words = rng.integers(32 if m.n_data_bits >= 7 else 0, 127 if m.n_data_bits >= 7 else 1 << m.n_data_bits,
                         40, dtype=np.uint32)
    clean = orc.tx_words(m, words, 1.0, 4096, True)
    spb = float(d.nsamples_per_bit)
    plan = orc.Plan(m.sample_rate, m.mark_f, m.space_f, m.band_width)
    nstreams = 192
    tmc = int(np.float32(np.float32(spb) * np.float32(0.75) + np.float32(0.5))) + d.nsamples_overscan
    wlen = pad4(tmc + d.expect_nsamples + int(spb) + 8)
    buf = np.zeros((nstreams, wlen), np.float32)
    first = d.nsamples_overscan
    for s in range(nstreams):
        sigma = (0.0, 0.0, 0.05, 0.3)[s % 4]
        pos = int(rng.integers(0, clean.size - wlen))
        buf[s] = (clean[pos:pos + wlen] + sigma * rng.standard_normal(wlen)).astype(np.float32)
    t = lambda a, dt: torch.from_numpy(np.ascontiguousarray(np.asarray(a).astype(dt))).to(dev())
    full = lambda v, dt: t(np.full(nstreams, v), dt)
    step = max(tmc // 8, 1)
    frames, mags = eng.find_frame_batch(t(buf, np.float32), full(wlen, np.int32), full(first, np.int32),
                                        full(tmc, np.int32), full(step, np.int32), full(np.inf, np.float32),
                                        bit_mags=True)
    torch.cuda.synchronize()
    fr = mm.frames_to_numpy(frames)
    mg = mags.cpu().numpy()
    eps = np.float32(1.1920928955078125e-07)
    n_checked = n_inf = 0
    for s in range(nstreams):
        if not fr[s]["confidence"] > 0:
            continue
        start = int(fr[s]["frame_start"])
        spb_fsk = float(np.float32(d.expect_nsamples) / np.float32(d.expect_n_bits))     # src/fsk.c:465
        c, bits, ampl, sig, noise, val = plan.frame_analyze(buf[s, start:].copy(), spb_fsk, d.expect_data)
        got_bits = int(fr[s]["bits_lo"]) | (int(fr[s]["bits_hi"]) << 32)
        assert got_bits == bits, (mode, s)
        avg = float(np.mean(sig))
        assert np.allclose(mg[s, :, 0], sig, rtol=1e-4, atol=0), (mode, s, mg[s, :, 0], sig)
        assert np.allclose(mg[s, :, 1], noise, rtol=0, atol=1e-4 * avg), (mode, s, mg[s, :, 1], noise)
        # the confidence=inf class: a noise magnitude at or below FLT_EPSILON is dropped from the sum (:279)
        assert np.array_equal(mg[s, :, 1] <= eps, noise <= eps), (mode, s, mg[s, :, 1], noise)
        n_inf += int((noise <= eps).any())
        n_checked += 1
    assert n_checked > nstreams // 4, n_checked
    if kw.get("space") == 2400:
        assert n_inf > 0            # the clean streams of this geometry do hit the class


# --------------------------------------------------------------------------
# every shipped rx kernel variant on hardware: the cp.async fill with the shared-segment search
# (default where the mode allows it) and with the per-candidate search, the TMA bulk fill
# (cp.async.bulk + mbarrier, FILL=1) and the warp-synchronous loop (FILL=3), each against the
# oracle on the same streams
# --------------------------------------------------------------------------
@pytest.mark.parametrize("variant", ["prefix", "prefix-cpasync", "multi", "multi-hybrid", "per-candidate", "tma-bulk", "warp-sync"])
@pytest.mark.parametrize("name", ["01-self-test-1200", "02-self-test-300", "small-rtty"])
def test_rx_kernel_variants_agree_with_the_oracle(name, variant, monkeypatch):
    env = {"prefix": {"FSK_B200_PREFIX": "1"},
           "prefix-cpasync": {"FSK_B200_PREFIX": "1", "FSK_B200_PFX_FILL": "0"},      # (what int16 rows and the emulator run)
           "multi": {"FSK_B200_MULTI": "2", "FSK_B200_PREFIX": "0"},
           "multi-hybrid": {"FSK_B200_MULTI": "1", "FSK_B200_PREFIX": "0"},
           "per-candidate": {"FSK_B200_MULTI": "0", "FSK_B200_PREFIX": "0"},
           "tma-bulk": {"FSK_B200_FILL": "1"}, "warp-sync": {"FSK_B200_FILL": "3"}}[variant]
    import conftest
    if variant == "tma-bulk" and conftest.EMU_DEVICE is not None:
        pytest.skip("the host emulation does not model cp.async.bulk / mbarrier")
    for k, v in env.items():
        monkeypatch.setenv(k, v)                # read when the engine is created
    case = refcases.BY_NAME[name]
    g = gu.load(case["name"])
    _, rx = gu.modes(case)
    a = gu.audio(case, g)
    eng, _ = engine_for(case)
    rng = np.random.default_rng(3)
    streams = [np.concatenate([np.zeros(int(rng.integers(0, 97)), np.float32), a]) for _ in range(9)]
    streams.append((a + 0.05 * rng.standard_normal(a.size)).astype(np.float32))
    recs, st = rx_on_gpu(eng, streams)
    kern = eng.last_kernel()
    if variant.startswith("prefix"):
        assert "prefix-table" in kern and ("fill=0" in kern) == (variant == "prefix-cpasync" or conftest.EMU_DEVICE is not None), kern
    elif variant.startswith("multi"):
        assert "shared-segment" in kern, kern
    elif variant == "per-candidate":
        assert "per-candidate" in kern, kern
    else:
        assert "fill=%s" % env["FSK_B200_FILL"] in kern, kern       # (FILL != 0 also keeps the prefix-table search out)
    for s, x in enumerate(streams):
        want = orc.rx_run(rx, x, literal=False)
        compare_frames(as_oracle_frames(recs[s]), want["frames"], "%s %s stream %d" % (name, variant, s))


# --------------------------------------------------------------------------
# the prefix-table kernel against the per-candidate kernel, frame by frame, far inside the oracle tolerance:
# the two form every window sum in a different order (chunk prefixes and their differences against one
# direct sum per window), so this is the per-window arithmetic of the new kernel checked to a few 1e-6 on
# noisy, offset and clean streams, the orthogonal-tone geometry (confidence = inf class) included
# --------------------------------------------------------------------------
@pytest.mark.parametrize("mode,kw,sigma", [
    ("300", {}, 0.0), ("300", {}, 0.2), ("rtty", dict(sample_rate=8000), 0.1), ("1200", {}, 0.3),
    ("same", {}, 0.05), ("1200", dict(mark=1200, space=2400), 0.0), ("300", dict(stopbits=2.0, startbits=2), 0.1)],
    ids=["bell103", "bell103-awgn", "rtty8k-awgn", "1200-awgn", "same-awgn", "orthogonal-tones", "300-2start-2stop"])
def test_prefix_table_kernel_against_the_per_candidate_kernel(mode, kw, sigma, monkeypatch):
    rx = orc.Mode(mode, **kw)
    d = rx.derived()
    rng = np.random.default_rng(77)
    streams = []
    for s in range(24):
        w = rng.integers(0, 1 << rx.n_data_bits, int(rng.integers(6, 30)), dtype=np.uint64).astype(np.uint32)
        x = np.concatenate([np.zeros(int(rng.integers(0, 4 * int(d.nsamples_per_bit))), np.float32),
                            orc.tx_words(rx, w, float(rng.uniform(0.2, 1.0)), 4096, True)]).astype(np.float32)
        if sigma:
            x = (x + np.float32(sigma * (0.5 + rng.random())) * rng.standard_normal(x.size).astype(np.float32)).astype(np.float32)
        if s % 5 == 4:
            x = (x - np.float32(0.07)).astype(np.float32)          # the reference's --Xrxnoise style offset
        streams.append(x)
    res = {}
    for variant, env in (("prefix", {"FSK_B200_PREFIX": "1"}), ("per-candidate", {"FSK_B200_PREFIX": "0", "FSK_B200_MULTI": "0"})):
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        eng, _ = engine_for((mode, kw))
        res[variant] = rx_on_gpu(eng, streams)
        assert ("prefix-table" in eng.last_kernel()) == (variant == "prefix"), eng.last_kernel()
        for k in env:
            monkeypatch.delenv(k)
    nframes = n_inf = 0
    for s in range(len(streams)):
        a, b = res["prefix"][0][s], res["per-candidate"][0][s]
        assert len(a) == len(b), (mode, s, len(a), len(b))
        for key in ("bits_lo", "bits_hi", "frame_start"):
            assert np.array_equal(a[key], b[key]), (mode, s, key)
        ca, cb = a["confidence"].astype(np.float64), b["confidence"].astype(np.float64)
        rep = a["frame_start"] == mm.FRAME_REPORT                    # (session reports carry sums, not confidences)
        inf = np.isinf(cb) & ~rep
        assert np.array_equal(np.isinf(ca) & ~rep, inf), (mode, s)
        fin = ~inf
        # a confidence is signal / noise: its sensitivity to the sums is ~confidence itself
        assert np.all(np.abs(ca[fin] - cb[fin]) <= 4e-6 * np.maximum(1.0, np.abs(cb[fin])) * np.abs(cb[fin]) + 1e-6), \
            (mode, s, float(np.max(np.abs(ca[fin] - cb[fin]) / np.maximum(np.abs(cb[fin]), 1e-9))))
        assert np.allclose(a["amplitude"], b["amplitude"], rtol=4e-6, atol=1e-7), (mode, s)
        nframes += int((~rep).sum())
        n_inf += int(inf.sum())
    assert nframes > 200, nframes
    if kw.get("space") == 2400 and not sigma:
        assert n_inf > 0


# --------------------------------------------------------------------------
# the BASELINE configurations at batch sizes of the bench's order (>= 16 384 streams each), generated
# on the device, a 1 % sample of the streams compared with the oracle frame by frame
# --------------------------------------------------------------------------
@pytest.mark.parametrize("mode,kw,nstreams,nwords,sigma", [
    ("1200", {}, 16384, 40, 0.0), ("1200", {}, 16384, 40, 0.35),
    ("rtty", dict(sample_rate=8000), 16384, 12, 0.0),
    ("300", {}, 16384, 12, 0.0), ("300", {}, 16384, 12, 0.25),
    ("same", {}, 16384, 24, 0.0)],
    ids=["cfg2", "cfg2-awgn", "cfg3-rtty8k", "cfg4-bell103", "cfg4-bell103-awgn", "cfg5-same"])
def test_baseline_configs_large_batch_sample_vs_oracle(mode, kw, nstreams, nwords, sigma):
    import conftest
    if conftest.EMU_DEVICE is not None:
        nstreams = 256                      # the host emulation is ~10^4 x slower
    m = orc.Mode(mode, **kw)
    d = m.derived()
    eng, cfg = engine_for((mode, kw))
    tcfg = mm.tx_config_from(cfg)
    gen = torch.Generator(device="cpu").manual_seed(5)
    mask = (1 << m.n_data_bits) - 1
    lo, hi = (32, 127) if m.n_data_bits >= 7 else (0, 1 << m.n_data_bits)
    words = (torch.randint(lo, hi, (nstreams, nwords), generator=gen, dtype=torch.int32) & mask)
    max_lead = 0 if cfg.do_rx_sync else max(1, int(d.nsamples_per_bit))
    lead = (torch.randint(0, max_lead, (nstreams,), generator=gen, dtype=torch.int32) if max_lead
            else torch.zeros(nstreams, dtype=torch.int32))
    n = int(orc.lib().orc_tx_nsamples(C.byref(m.tx_config(1.0, 4096, True)), nwords)) + max_lead + 64
    x = mm.tx_batch(tcfg, words.to(dev()), n, lead_in=lead.to(dev()))
    if sigma:
        g2 = torch.Generator(device="cpu").manual_seed(6)
        x = x + (sigma * torch.randn(x.shape, generator=g2, dtype=torch.float32)).to(dev())
        x = x.contiguous()
    frames, states = eng.rx_batch(x, nsamples=n)
    torch.cuda.synchronize()
    # the default policy: shared-segment search where the bit period is long and the windows tile
    if not (os.environ.get("FSK_B200_PREFIX") or os.environ.get("FSK_B200_MULTI")):      # the defaults, unless a run forces a variant
        assert ("shared-segment" in eng.last_kernel() or "prefix-table" in eng.last_kernel()) == (mode in ("rtty", "300")), eng.last_kernel()
    st = mm.states_to_numpy(states)
    assert (st["done"] == 1).all()
    rows = np.arange(0, nstreams, max(1, nstreams // max(8, nstreams // 100)))
    fr = mm.frames_to_numpy(frames[torch.from_numpy(rows).to(dev())])
    hx = x[torch.from_numpy(rows).to(dev())].cpu().numpy()
    n_flip = 0
    for i, s in enumerate(rows):
        want = orc.rx_run(m, hx[i, :n].copy(), literal=False)
        got = as_oracle_frames(fr[i, :st["nframes"][s]])
        try:
            compare_frames(got, want["frames"], "%s stream %d" % (mode, s))
        except AssertionError:
            assert sigma > 0, (mode, s)         # clean streams: exact
            n_flip += 1
            assert [orc.databits(m, f[0]) for f in got][:4] == [orc.databits(m, f[0]) for f in want["frames"]][:4]
    assert n_flip <= max(1, len(rows) // 50), (n_flip, len(rows))


# --------------------------------------------------------------------------
# N2 fused: int16 PCM rows resident in HBM, widened inside the rx kernel's ring fill
# (fsk_b200_rx_batch_s16) -- the records must be those of the float path on short/32768, bit for bit
# --------------------------------------------------------------------------
@pytest.mark.parametrize("mode,kw", [("1200", {}), ("300", {}), ("rtty", dict(sample_rate=8000)), ("same", {}),
                                     ("0.5", dict(sample_rate=8000))],
                         ids=["1200", "bell103", "rtty8k", "same", "generic-0.5baud"])
def test_rx_batch_s16_resident_is_bit_identical_to_the_float_path(mode, kw):
    m = orc.Mode(mode, **kw)
    eng, cfg = engine_for((mode, kw))
    rng = np.random.default_rng(16)
    nstreams = 21
    nwords = 3 if mode == "0.5" else 30
    rows, lens = [], []
    for s in range(nstreams):
        lo, hi = (32, 127) if m.n_data_bits >= 7 else (0, 1 << m.n_data_bits)
        words = rng.integers(lo, hi, nwords, dtype=np.uint32)
        x = orc.tx_words(m, words, 0.8, 4096, False)        # the transmitter's int16 samples, as floats / 32768
        lead = 0 if cfg.do_rx_sync else int(rng.integers(0, 200))
        x = np.concatenate([np.zeros(lead, np.float32), x, np.zeros(int(rng.integers(0, 300)), np.float32)])
        if s % 5 == 4:
            x = x[: x.size * 2 // 3]                       # ragged: cut in mid frame
        rows.append(np.round(x * 32768.0).astype(np.int16))
        lens.append(x.size)
    n = max(lens)
    stride = (n + 7) & ~7
    pcm = np.zeros((nstreams, stride), np.int16)
    for s, r in enumerate(rows):
        pcm[s, :r.size] = r
    lens_t = torch.from_numpy(np.asarray(lens, np.int32)).to(dev())
    d16 = torch.from_numpy(pcm).to(dev())
    f32 = mm.s16_to_f32(d16)
    fr_a, st_a = eng.rx_batch(f32, nsamples=n, nsamples_each=lens_t)
    fr_b, st_b = eng.rx_batch(d16, nsamples=n, nsamples_each=lens_t)
    torch.cuda.synchronize()
    assert "src=s16" in eng.last_kernel(), eng.last_kernel()
    sa, sb = mm.states_to_numpy(st_a), mm.states_to_numpy(st_b)
    for f in ("pos", "nframes", "carrier", "noconfidence", "done", "carrier_nsamples", "nframes_decoded"):
        assert np.array_equal(sa[f], sb[f]), f
    assert sa["nframes"].sum() > nstreams * (2 if mode == "0.5" else 10)
    a, b = mm.frames_to_numpy(fr_a), mm.frames_to_numpy(fr_b)
    for s in range(nstreams):
        k = int(sa["nframes"][s])
        assert a[s, :k].tobytes() == b[s, :k].tobytes(), (mode, s)
    # resumed from a position that is not a multiple of 8 (the int16 fill aligns to 16 bytes = 8 samples)
    st_c = st_b.clone()
    st_c.zero_()
    sc = mm.states_to_numpy(st_c).copy()
    sc["pos"][:] = 13
    st_c = torch.from_numpy(sc.view(np.int32).reshape(nstreams, -1)).to(dev())
    st_d = st_c.clone()
    fr_c, st_c = eng.rx_batch(f32, nsamples=n, nsamples_each=lens_t, states=st_c)
    fr_d, st_d = eng.rx_batch(d16, nsamples=n, nsamples_each=lens_t, states=st_d)
    torch.cuda.synchronize()
    c, d = mm.frames_to_numpy(fr_c), mm.frames_to_numpy(fr_d)
    sc2 = mm.states_to_numpy(st_c)
    for s in range(nstreams):
        k = int(sc2["nframes"][s])
        assert c[s, :k].tobytes() == d[s, :k].tobytes(), (mode, s, "resumed")


def test_live_receiver_frames_with_three_stop_bits_in_tiny_chunks():
    """ADVICE (round 1): with 2.5 or more stop bits a frame's advance (frame_start + frame_nsamples - overscan,
    src/minimodem.c:1407) exceeds the search window, and a hold-back sized for the window alone let an
    iteration record its frame, hit the end-of-input exit of :1151 and be replayed after the next chunk:
    the frame came out twice.  fsk_b200_stream_window now covers the largest advance; chunks of at most
    40 samples must give the text of one pass over the whole stream."""
    case = refcases.BY_NAME["more-150-stop3"]
    g = gu.load(case["name"])
    _, rx = gu.modes(case)
    a = gu.audio(case, g)
    names = dict(mark="f_mark", space="f_space", bandwidth="band_width", startbits="nstartbits", stopbits="nstopbits")
    ov = {names.get(k, k): v for k, v in case["rx_mkw"].items() if k != "sample_rate"}
    # one pass over the complete stream (the batched, flat-buffer semantic: the reference's own ring stops
    # after the first frame of this vector, DESIGN.md 5.2, so its stdout is only a prefix of this)
    eng, _ = engine_for(case)
    buf = np.zeros((1, pad4(a.size)), np.float32)
    buf[0, :a.size] = a
    frames, states = eng.rx_batch(torch.from_numpy(buf).to(dev()), nsamples=a.size)
    out, cnt = eng.decode_batch(mm.decoder_for_mode(case["rx_mode"], rx.n_data_bits), frames, states)
    torch.cuda.synchronize()
    want = bytes(out.cpu().numpy()[0, :int(cnt.cpu().numpy()[0])])
    assert want.startswith(bytes(g["stdout"])) and len(want) > 8, want
    rng = np.random.default_rng(5)
    nstreams, max_chunk = 3, 40
    lr = mm.LiveReceiver(case["rx_mode"], sample_rate=rx.sample_rate, nstreams=nstreams, max_chunk=max_chunk,
                         device=dev(), **ov)
    fed = [0] * nstreams
    text = [bytearray() for _ in range(nstreams)]

    def take(o, c):
        o, c = o.cpu().numpy(), c.cpu().numpy()
        for i in range(nstreams):
            text[i] += bytes(o[i, :c[i]])

    while any(f < a.size for f in fed):
        chunk = np.zeros((nstreams, max_chunk), np.float32)
        clen = np.zeros(nstreams, np.int32)
        for i in range(nstreams):
            k = int(min(rng.integers(1, max_chunk + 1) if i else max_chunk, a.size - fed[i]))
            chunk[i, :k] = a[fed[i]:fed[i] + k]
            clen[i] = k
            fed[i] += k
        take(*lr.feed(torch.from_numpy(chunk).to(dev()), torch.from_numpy(clen).to(dev())))
    take(*lr.finish())
    torch.cuda.synchronize()
    for i in range(nstreams):
        assert bytes(text[i]) == want, (i, bytes(text[i]), want)
