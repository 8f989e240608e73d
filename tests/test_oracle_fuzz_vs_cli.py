"""Differential fuzz of the oracle against the UNMODIFIED reference CLI (oracle/_ref/minimodem_ref; its
recorded answers, tests/golden/reference_results.json, where it is not built): random baud rates, sample
rates, framings, bit orders, tone pairs and payloads go through the reference's own transmitter and
receiver; the oracle's transmitter must produce the same samples, and the oracle's rx loop (LITERAL mode,
the reference's ring and all) the same text and the same stat lines.  The golden vectors pin fixed cases;
this pins the space between them."""
import hashlib

import numpy as np
import pytest

import golden_util as gu
import orc


def random_invocation(rng):
    while True:
        baud = int(rng.choice([75, 110, 150, 300, 600, 1200, 2400, 4800]))
        rate = int(rng.choice([8000, 11025, 16000, 22050, 44100, 48000]))
        if not (6 <= rate / baud <= 700):
            continue
        args, kw = [str(baud), "--samplerate", str(rate)], dict(sample_rate=rate)
        if rng.random() < 0.3:
            args = ["-7"] + args
            kw["n_data_bits"] = 7
        if rng.random() < 0.4:
            sb = int(rng.choice([1, 2, 3]))
            args += ["--startbits", str(sb)]
            kw["startbits"] = sb
        if rng.random() < 0.5:
            st = float(rng.choice([1.0, 1.5, 2.0]))
            args += ["--stopbits", str(st)]
            kw["stopbits"] = st
        for flag, key in (("--msb-first", "msb_first"), ("--invert-start-stop", "invert_start_stop"),
                          ("--inverted", "inverted")):
            if rng.random() < 0.25:
                args.append(flag)
                kw[key] = True
        if rng.random() < 0.3 and baud >= 400:
            mark = float(rng.choice([1000, 1300, 1500, 1800]))
            space = mark + float(rng.choice([400, 600, 1000]))
            if space < rate / 2 - 300:
                args += ["-M", str(mark), "-S", str(space)]
                kw["mark"], kw["space"] = mark, space
        flt = rng.random() < 0.3
        vol = float(rng.choice([1.0, 0.5, 0.1]))
        tx = args + (["--float-samples"] if flt else []) + (["--volume", str(vol)] if vol != 1.0 else [])
        try:
            m = orc.Mode(str(baud), **kw)
            m.derived()
            orc.Plan(m.sample_rate, m.mark_f, m.space_f, m.band_width)
        except Exception:
            continue
        if m.frame_n_bits > 12:            # longer frames hit the reference's ring limit (DESIGN.md 5, item 2)
            continue
        return str(baud), kw, tx, args, flt, vol


@pytest.mark.parametrize("seed", range(60))
def test_oracle_matches_the_reference_cli_on_a_random_invocation(seed):
    rng = np.random.default_rng(5000 + seed)
    mode, kw, tx_args, rx_args, flt, vol = random_invocation(rng)
    text = bytes(rng.integers(32, 127, int(rng.integers(4, 40)), dtype=np.uint8)) + b"\n"
    r = orc.ref_cli(tx_args, rx_args, text)
    m = orc.Mode(mode, **kw)
    # the transmitter restatement: same samples
    words = orc.ref_encode("ascii8", text) & ((1 << m.n_data_bits) - 1)
    audio = orc.tx_words(m, words, vol, 4096, flt)
    assert audio.size == r["audio_len"], (tx_args, audio.size, r["audio_len"])
    assert hashlib.sha256(audio.tobytes()).hexdigest() == r["audio_sha256"], tx_args
    # the rx loop restatement, with the reference's ring: same text, same stat lines
    res = orc.rx_run(m, audio, literal=True)
    assert orc.ref_decode(m, res["frames"]) == r["stdout"], (rx_args, r["stdout"][:40])
    want = r["nocarrier"]
    got = [orc.report_line(m, rp) for rp in res["reports"]]
    assert len(got) == len(want), (rx_args, got, want)
    for a_line, b_line in zip(got, want):
        fa, fb = a_line.split(), b_line.split()
        assert fa[:3] == fb[:3] and fa[4:] == fb[4:], (a_line, b_line)
        assert gu.close(float(fa[3].split("=")[1]), float(fb[3].split("=")[1]), 2e-3, cond=gu.CONF_COND)
