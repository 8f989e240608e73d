"""Pin the oracle's bit analyzer / frame search against (a) the raw FFT bins the
unmodified reference computed on its own vectors (tests/golden, `bins`) and
(b) oracle/_ref/libfsk_ref.so = the unmodified src/fsk.c compiled in place, on
seeded noisy inputs (its recorded answers where it is not built).  CPU only."""
import numpy as np
import pytest

import golden_util as gu
import orc
import refcases

BIN_CASES = [c for c in refcases.ALL if c["bins"]]


@pytest.mark.parametrize("case", BIN_CASES, ids=[c["name"] for c in BIN_CASES])
def test_two_bin_dft_matches_reference_fft_bins(case):
    """Replay every bit window the reference analysed (same scan order, same
    two-pass order, same early rejects) and compare magnitudes with its FFT."""
    g = gu.load(case["name"])
    _, rx = gu.modes(case)
    a = gu.audio(case, g)
    if case["rxnoise"]:
        a = a + np.float32(-0.5) * np.float32(case["rxnoise"] * 2)
    r = orc.rx_run(rx, a, literal=True, rxnoise=0.0, rx_one=case["rx_one"], want_calls=True)
    plan = orc.Plan(rx.sample_rate, rx.mark_f, rx.space_f, rx.band_width)
    bins = g["bins"]
    nfft = g["call_nfft"]
    assert len(r["calls"]) == len(nfft)
    apad = np.concatenate([a, np.zeros(1 << 16, np.float32)])
    k = 0
    worst_sig, worst_noise = 0.0, 0.0
    # The reference refills its ring only below half full (src/minimodem.c:1158), yet
    # fsk_find_frame may touch try_max-1+span samples; for slow modes (< ~288 baud at
    # 48 kHz) that exceeds the guaranteed-valid half and it reads STALE ring contents.
    # Those windows are not comparable with a flat buffer (DESIGN.md, "stale reads").
    half = rx.derived().samplebuf_size // 2
    n_stale = 0
    for ci, c in enumerate(r["calls"]):
        frame_nsamples, try_first, try_max, try_step, limit, use_sync, conf, bits, ampl, start, pos = c
        expect = bytes(g["call_expect"][ci])
        n_bits = len(expect)
        spb = np.float32(frame_nsamples) / np.float32(n_bits)
        N = int(np.float32(spb + np.float32(0.5)))
        scalar = np.float32(2.0) / np.float32(N)
        kend = k + int(nfft[ci])
        j = 0
        best = np.float32(0)
        while k < kend:
            up = 1 if j % 2 else -1
            t = try_first + up * ((j + 1) // 2) * try_step
            j += 1
            if t >= try_max:
                break
            if t < 0:
                continue
            order = [b for b in range(n_bits) if expect[b] != ord("d")] + \
                    [b for b in range(n_bits) if expect[b] == ord("d")]
            rejected = False
            for b in order:
                begin = int(np.float32(spb * np.float32(b) + np.float32(0.5)))
                w = apad[pos + t + begin: pos + t + begin + N]
                mm, ms = plan.bit_mags(np.ascontiguousarray(w), N)
                rm = np.float32(np.hypot(bins[k, 0], bins[k, 1])) * scalar
                rs = np.float32(np.hypot(bins[k, 2], bins[k, 3])) * scalar
                k += 1
                hi, lo = max(rm, rs), min(rm, rs)
                ohi, olo = max(mm, ms), min(mm, ms)
                if t + begin + N > half:
                    n_stale += 1
                elif hi > 0:
                    worst_sig = max(worst_sig, abs(float(ohi) - float(hi)) / float(hi))
                    worst_noise = max(worst_noise, abs(float(olo) - float(lo)) / float(hi))
                if expect[b] != ord("d") and (1 if rm > rs else 0) != expect[b] - ord("0"):
                    rejected = True
                    break
            if rejected:
                continue
    assert k == len(bins)
    assert n_stale <= len(bins) // 50
    # the reference's own float FFT carries ~1e-7 relative error per bin
    assert worst_sig < 2e-6, worst_sig
    assert worst_noise < 2e-6, worst_noise


@pytest.mark.parametrize("mode_name,kw", [("1200", {}), ("300", {}), ("rtty", dict(sample_rate=8000)),
                                          ("same", {}), ("12000", {}), ("rtty", {})])
def test_find_frame_matches_compiled_reference_on_noisy_input(mode_name, kw):
    m = orc.Mode(mode_name, **kw)
    d = m.derived()
    rng = np.random.default_rng(1234)
    words = rng.integers(0, 1 << m.n_data_bits, 24, dtype=np.uint32)
    clean = orc.tx_words(m, words, 1.0, 4096, True)
    plan = orc.Plan(m.sample_rate, m.mark_f, m.space_f, m.band_width)
    rplan = orc.RefPlan(m.sample_rate, m.mark_f, m.space_f, m.band_width)
    spb = float(d.nsamples_per_bit)
    n_checked = n_found = n_bad = 0
    for sigma in (0.0, 0.1, 0.5, 1.0):
        a = (clean + sigma * rng.standard_normal(clean.size)).astype(np.float32)
        a = np.concatenate([a, np.zeros(4 * int(spb) + d.expect_nsamples, np.float32)])
        for trial in range(40):
            pos = int(rng.integers(0, clean.size - d.expect_nsamples))
            carrier = trial % 2
            try_max = int(np.float32(np.float32(spb) * np.float32(0.75) + np.float32(0.5))) if carrier else int(spb)
            try_max += d.nsamples_overscan
            fine = (trial // 2) % 2
            step = max(try_max // (8 if fine else 3), 1)
            limit = np.inf if fine else 2.3
            first = d.nsamples_overscan if carrier else 0
            expect = d.expect_data if carrier else d.expect_sync
            w = np.ascontiguousarray(a[pos: pos + try_max + d.expect_nsamples + int(spb) + 2])
            got = plan.find_frame(w, d.expect_nsamples, first, try_max, step, limit, expect)
            want = rplan.find_frame(w, d.expect_nsamples, first, try_max, step, limit, expect)
            n_checked += 1
            n_found += want[0] > 0
            # decisions are float comparisons; on noisy data a tie-level difference
            # between two correct DFTs may legitimately pick another candidate,
            # so require exact agreement only when the result is not razor-edge.
            ok = (got[1] == want[1] and got[3] == want[3]
                  and gu.close(got[0], want[0], cond=gu.CONF_COND) and gu.close(got[2], want[2]))
            if not ok:
                n_bad += 1
                assert sigma > 0, (mode_name, sigma, trial, got, want)
    assert n_found > n_checked // 8
    assert n_bad <= 1, n_bad      # razor-edge candidate flips only


@pytest.mark.ref
@pytest.mark.parametrize("mode,kw", [("1200", {}), ("300", {}), ("rtty", dict(sample_rate=8000)), ("same", {})])
def test_dfti_backed_reference_build_agrees_with_the_portable_one(mode, kw):
    """oracle/_ref/libfsk_ref_dfti.so (the unmodified src/fsk.c on MKL's FFT, used only to time the
    reference fairly in bench.py) against oracle/_ref/libfsk_ref.so (the same source on the portable
    FFT stand-in, which minted the golden vectors): same searches, same bits and frame starts,
    confidences equal to FFT rounding."""
    if not orc.have_ref_dfti():
        pytest.skip("libfsk_ref_dfti.so not built (needs PyTorch's libtorch_cpu.so)")
    import ctypes as C
    m = orc.Mode(mode, **kw)
    d = m.derived()
    A, B = orc.ref(), orc.ref_dfti()
    rng = np.random.default_rng(12)
    a = orc.tx_words(m, rng.integers(0, 1 << m.n_data_bits, 40, dtype=np.uint32), 0.8, 4096, True)
    a = (a + np.float32(0.05) * rng.standard_normal(a.size).astype(np.float32)).astype(np.float32)
    a = np.concatenate([a, np.zeros(4 * d.expect_nsamples, np.float32)])
    pa = A.fsk_plan_new(m.sample_rate, m.mark_f, m.space_f, m.band_width)
    pb = B.fsk_plan_new(m.sample_rate, m.mark_f, m.space_f, m.band_width)
    assert pa and pb
    try_max = int(d.nsamples_per_bit) + d.nsamples_overscan
    n_checked = 0
    for pos in range(0, a.size - 3 * d.expect_nsamples, max(1, d.expect_nsamples // 3)):
        w = np.ascontiguousarray(a[pos:pos + 3 * d.expect_nsamples])
        res = []
        for L, p in ((A, pa), (B, pb)):
            bits, ampl, start = C.c_ulonglong(0), C.c_float(0), C.c_uint(0)
            c = L.fsk_find_frame(p, orc.fptr(w), d.expect_nsamples, 0, try_max, max(1, try_max // 8),
                                 float("inf"), d.expect_data, C.byref(bits), C.byref(ampl), C.byref(start))
            res.append((np.float32(c), bits.value, np.float32(ampl.value), start.value))
        (ca, ba, aa, sa), (cb, bb, ab, sb) = res
        if ba == bb and sa == sb:
            assert gu.close(ca, cb, 1e-4, cond=gu.CONF_COND) and gu.close(aa, ab)
            n_checked += 1
        else:
            # two float FFTs may prefer different candidates only when those are equal to rounding
            assert gu.close(ca, cb, 1e-3, cond=gu.CONF_COND), (pos, res)
    assert n_checked > 20
    A.fsk_plan_destroy(pa)
    B.fsk_plan_destroy(pb)
