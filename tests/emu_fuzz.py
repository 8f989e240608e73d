"""Random modes through the emulated kernels (run by tests/test_emu_parity.py in a subprocess with
FSK_B200_EMU=1; the file name keeps pytest from collecting it on its own).

Framings, bit orders, rates and baud rates that no committed vector has: the oracle's transmitter
makes the stream, the oracle's rx loop says what the records must be, the kernels' source (on the
host SIMT emulator) has to produce them -- exact bits, frame starts and acquire flags, confidence
and amplitude to the parity tolerance.  This is a logic check of the kernels over geometry the
vectors do not reach (window counts from 7 to 44 bits, every lane split the launcher picks,
fractional samples per bit, long windows); it runs on the emulator only, because a near-tie that
the B200's approximate divide resolves the other way would make a random case flaky there."""
import numpy as np
import pytest

import minimodem_b200 as mm
import orc
import test_gpu_parity as T

pytestmark = pytest.mark.gpu

BAUDS = [75, 110, 150, 300, 600, 1200, 2400, 4800]
RATES = [8000, 11025, 16000, 22050, 44100, 48000]


def random_mode(rng):
    while True:
        baud = int(rng.choice(BAUDS))
        rate = int(rng.choice(RATES))
        spb = rate / baud
        if spb < 6 or spb > 700:
            continue
        kw = dict(sample_rate=rate)
        kw["n_data_bits"] = int(rng.choice([5, 6, 7, 8, 9, 12, 16, 24, 32]))
        kw["startbits"] = int(rng.choice([1, 1, 2, 3, 5]))
        kw["stopbits"] = float(rng.choice([1.0, 1.0, 1.5, 2.0, 3.0]))
        kw["msb_first"] = bool(rng.integers(0, 2))
        kw["invert_start_stop"] = bool(rng.integers(0, 2))
        kw["inverted"] = bool(rng.integers(0, 2))
        if kw["n_data_bits"] + kw["startbits"] + kw["stopbits"] + 1 > 48:
            continue
        try:
            m = orc.Mode(str(baud), **kw)
            m.derived()
            orc.Plan(m.sample_rate, m.mark_f, m.space_f, m.band_width)
        except Exception:
            continue
        if max(m.mark_f, m.space_f) >= rate / 2 - m.band_width:
            continue
        return str(baud), kw


@pytest.mark.parametrize("seed", range(64))
def test_random_mode_records_match_the_oracle(seed):
    rng = np.random.default_rng(1000 + seed)
    mode, kw = random_mode(rng)
    rx = orc.Mode(mode, **kw)
    nwords = int(rng.integers(6, 18))
    words = rng.integers(0, 1 << rx.n_data_bits, nwords, dtype=np.uint64).astype(np.uint32)
    streams = []
    for s in range(3):
        a = orc.tx_words(rx, words, float(rng.uniform(0.3, 1.0)), 4096, True)
        lead = int(rng.integers(0, 3 * int(rx.derived().nsamples_per_bit) + 1))
        x = np.concatenate([np.zeros(lead, np.float32), a])
        x = (x + np.float32(0.01) * rng.standard_normal(x.size).astype(np.float32)).astype(np.float32)
        streams.append(x)
    eng, _ = T.engine_for((mode, kw))
    recs, st = T.rx_on_gpu(eng, streams)
    decoded = 0
    for s, x in enumerate(streams):
        want = orc.rx_run(rx, x, literal=False)
        got = T.as_oracle_frames(recs[s])
        T.compare_frames(got, want["frames"], "%s %r stream %d" % (mode, kw, s))
        T.compare_reports(T.reports_of(recs[s], st[s]), want["reports"], "%s %r stream %d" % (mode, kw, s))
        decoded += len(got)
    assert decoded >= nwords, (mode, kw, decoded, nwords)


STRESS_MODES = [("1200", {}), ("300", {}), ("rtty", dict(sample_rate=8000)), ("same", {}),
                ("2400", dict(sample_rate=44100)), ("110", dict(sample_rate=11025, stopbits=2.0))]


@pytest.mark.parametrize("mi", range(len(STRESS_MODES)))
@pytest.mark.parametrize("seed", range(4))
def test_dropouts_bursts_and_resume(mi, seed):
    """Streams that keep losing and finding the carrier: bursts of frames separated by silence,
    noise and truncated frames of random lengths (ring restarts, the 20-strike carrier drop,
    session reports), decoded once in one go and once in record buffers of a few frames with
    the saved state carried over -- both must equal the oracle's rx loop."""
    mode, kw = STRESS_MODES[mi]
    rx = orc.Mode(mode, **kw)
    rng = np.random.default_rng(7000 + 10 * mi + seed)
    spb = int(rx.derived().nsamples_per_bit)
    streams = []
    for s in range(4):
        parts = []
        for _ in range(int(rng.integers(2, 5))):
            kind = int(rng.integers(0, 4))
            gap = int(rng.integers(1, 60)) * spb + int(rng.integers(0, spb))
            if kind == 0:
                parts.append(np.zeros(gap, np.float32))
            elif kind == 1:
                parts.append((0.2 * rng.standard_normal(gap)).astype(np.float32))
            words = rng.integers(0, 1 << rx.n_data_bits, int(rng.integers(2, 12)), dtype=np.uint64).astype(np.uint32)
            a = orc.tx_words(rx, words, float(rng.uniform(0.2, 1.0)), 4096, True)
            if kind == 3:
                a = a[:int(rng.integers(a.size // 3, a.size))]      # cut inside a frame
            parts.append(a)
        x = np.concatenate(parts).astype(np.float32)
        x = (x + np.float32(0.003) * rng.standard_normal(x.size).astype(np.float32)).astype(np.float32)
        streams.append(x)
    eng, _ = T.engine_for((mode, kw))
    recs, st = T.rx_on_gpu(eng, streams)
    wants = [orc.rx_run(rx, x, literal=False) for x in streams]
    for s in range(len(streams)):
        T.compare_frames(T.as_oracle_frames(recs[s]), wants[s]["frames"], "%s stream %d" % (mode, s))
        T.compare_reports(T.reports_of(recs[s], st[s]), wants[s]["reports"], "%s stream %d" % (mode, s))

    # the same in record buffers of 3 frames, resumed until every stream is done
    torch = T.torch
    n = max(len(a) for a in streams)
    buf = np.zeros((len(streams), T.pad4(n)), np.float32)
    for i, a in enumerate(streams):
        buf[i, :len(a)] = a
    d = torch.from_numpy(buf).to(T.dev())
    lens = torch.from_numpy(np.array([len(a) for a in streams], np.int32)).to(T.dev())
    states = None
    got = [[] for _ in streams]
    for _ in range(400):
        frames, states = eng.rx_batch(d, nsamples=n, nsamples_each=lens, max_frames=3, states=states)
        fr, s1 = mm.frames_to_numpy(frames), mm.states_to_numpy(states)
        for i in range(len(streams)):
            got[i].extend(fr[i, :s1["nframes"][i]].copy())
        if (s1["done"] == 1).all():
            break
        # the binding hands the state back; the record count starts over for the next buffer
        s2 = s1.copy()
        s2["nframes"] = 0
        states = torch.from_numpy(s2.view(np.int32).reshape(len(streams), -1)).to(T.dev())
    else:
        raise AssertionError("streams did not finish")
    for i in range(len(streams)):
        T.compare_frames(T.as_oracle_frames(got[i]), wants[i]["frames"], "%s stream %d resumed" % (mode, i))


import refcases  # noqa: E402


@pytest.mark.parametrize("case", refcases.MORE, ids=[c["name"] for c in refcases.MORE])
def test_second_batch_of_option_vectors(case):
    """tests/refcases.py MORE: runs of the unmodified reference CLI that are on the CPU lists only;
    here the emulated kernels have to reproduce their records, decoded bytes and stat lines."""
    if case["ring_limited"]:
        # the kernels follow the flat semantic: all of the text, of which the reference printed the start
        g = T.gu.load(case["name"])
        _, rx = T.gu.modes(case)
        a = T.gu.audio(case, g)
        eng, _ = T.engine_for(case)
        (recs,), st = T.rx_on_gpu(eng, [a])
        got = T.as_oracle_frames(recs)
        T.compare_frames(got, orc.rx_run(rx, a, literal=False)["frames"], case["name"])
        out = orc.decode_records(rx, refcases.decoder_of(case, rx), orc.frame_records(got))
        assert out == bytes(g["text"]) and out.startswith(bytes(g["stdout"]))
        return
    T.test_rx_batch_on_reference_vectors(case)


@pytest.mark.parametrize("seed", range(40))
def test_batched_kernels_print_what_the_reference_cli_prints(seed):
    """Closing the loop without the oracle in between: a random invocation goes through the
    unmodified reference CLI (transmit, then receive; its recorded answers where oracle/_ref is not
    built), and the same audio through rx_batch + decode_batch on the emulated kernels; the text must
    be the CLI's stdout.  (Where the reference's sample ring makes it read stale samples -- slow
    modes, DESIGN.md 5 item 2 -- the oracle's two modes already differ and the case is skipped.)"""
    import hashlib
    from test_oracle_fuzz_vs_cli import random_invocation
    rng = np.random.default_rng(12000 + seed)
    mode, kw, tx_args, rx_args, flt, vol = random_invocation(rng)
    text = bytes(rng.integers(32, 127, int(rng.integers(4, 30)), dtype=np.uint8)) + b"\n"
    ref = orc.ref_cli(tx_args, rx_args, text)
    m = orc.Mode(mode, **kw)
    # the audio the reference's transmitter wrote, from the oracle's bit-exact restatement of it
    audio = orc.tx_words(m, orc.ref_encode("ascii8", text) & ((1 << m.n_data_bits) - 1), vol, 4096, flt)
    assert hashlib.sha256(audio.tobytes()).hexdigest() == ref["audio_sha256"], tx_args
    lit = orc.rx_run(m, audio, literal=True)["frames"]
    flat = orc.rx_run(m, audio, literal=False)["frames"]
    if [f[:1] + f[3:5] for f in lit] != [f[:1] + f[3:5] for f in flat]:
        pytest.skip("the reference's ring changes this one")
    eng, _ = T.engine_for((mode, kw))
    n = audio.size
    buf = np.zeros((2, T.pad4(n)), np.float32)
    buf[:, :n] = audio
    frames, states = eng.rx_batch(T.torch.from_numpy(buf).to(T.dev()), nsamples=n)
    out, cnt = eng.decode_batch(mm.decoder_for_mode(mode, m.n_data_bits), frames, states)
    o, c = out.cpu().numpy(), cnt.cpu().numpy()
    for s in range(2):
        assert bytes(o[s, :c[s]]) == ref["stdout"], (rx_args, bytes(o[s, :c[s]])[:40], ref["stdout"][:40])
