"""Pin the oracle (oracle/fsk_oracle.c) against the golden vectors minted from
the UNMODIFIED reference CLI (tests/golden/make_golden.py): TX restatement is
bit-exact, the rx-loop restatement reproduces every fsk_find_frame call, the
decoded bytes and the NOCARRIER stat lines.  CPU only."""
import numpy as np
import pytest

import golden_util as gu
import orc
import refcases

CASES = refcases.EVERY + refcases.MORE
IDS = [c["name"] for c in CASES]


@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_tx_restatement_bit_exact(case):
    g = gu.load(case["name"])
    tx, _ = gu.modes(case)
    a = orc.tx_words(tx, g["words"], case["amplitude"], case["lut"], case["float_samples"])
    assert a.size == int(g["audio_len"][0])
    assert gu.sha(a) == bytes(g["audio_sha256"])


@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_rx_restatement_matches_reference_calls(case):
    g = gu.load(case["name"])
    _, rx = gu.modes(case)
    a = gu.audio(case, g)
    r = orc.rx_run(rx, a, literal=True, rxnoise=case["rxnoise"], rx_one=case["rx_one"], want_calls=True)
    cu, cf, cb = g["call_u32"], g["call_f32"], g["call_bits"]
    assert len(r["calls"]) == len(cb)
    d = rx.derived()
    for i, c in enumerate(r["calls"]):
        frame_nsamples, try_first, try_max, try_step, limit, use_sync, conf, bits, ampl, start, pos = c
        assert (frame_nsamples, try_first, try_max, try_step) == tuple(int(x) for x in cu[i, :4]), i
        assert np.float32(limit) == cf[i, 0] or (np.isinf(limit) and np.isinf(cf[i, 0])), i
        exp = d.expect_sync if use_sync else d.expect_data
        assert exp == bytes(g["call_expect"][i]), i
        assert bits == int(cb[i]), (i, hex(bits), hex(int(cb[i])))
        assert start == int(cu[i, 4]), i
        assert gu.close(conf, cf[i, 1], cond=gu.CONF_COND), (i, conf, cf[i, 1])
        assert gu.close(ampl, cf[i, 2]), (i, ampl, cf[i, 2])


@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_rx_restatement_decodes_and_reports_like_reference(case):
    g = gu.load(case["name"])
    _, rx = gu.modes(case)
    a = gu.audio(case, g)
    for literal in (True, False):
        r = orc.rx_run(rx, a, literal=literal, rxnoise=case["rxnoise"], rx_one=case["rx_one"])
        out = orc.ref_decode(rx, r["frames"], decoder=refcases.decoder_of(case, rx))
        if case["ring_limited"] and not literal:
            # the reference gave up early (its ring); the flat semantic goes on: same beginning, more text
            assert out.startswith(bytes(g["stdout"])) and len(out) > len(bytes(g["stdout"]))
            assert out == bytes(g["text"])
            continue
        assert out == bytes(g["stdout"]), ("literal" if literal else "flat")
        want = gu.stat_lines(g)
        got = [orc.report_line(rx, rp) for rp in r["reports"]]
        if case["rx_one"]:
            got = got[:1]
        # ill-conditioned confidences (noise ~ 0, SURVEY hard part 3) may differ in the
        # printed decimals; everything else must be identical text
        assert len(got) == len(want)
        for a_line, b_line in zip(got, want):
            fa, fb = a_line.split(), b_line.split()
            assert fa[:3] == fb[:3] and fa[4:] == fb[4:], (a_line, b_line)
            ca, cb = float(fa[3].split("=")[1]), float(fb[3].split("=")[1])
            assert gu.close(ca, cb, 2e-3, cond=gu.CONF_COND), (a_line, b_line)
